#!/usr/bin/env python
"""bench.py -- headline benchmark of the Agilex-NTT hot path on B200.

Metric (BASELINE.json): NTT+INTT pairs/sec at n=4096, one 30-bit prime, batch of 65,536 polynomials per GPU
(configs[1]); a "step" is one forward launch + one inverse launch over the whole 1 GiB batch, in place, inputs
resident in HBM.  Multi-GPU: one process per GPU (torchrun), the batch dimension is sharded with no data-path
collective (weak scaling: 65,536 polynomials per GPU); the only collectives are the barrier, the max-over-ranks
reduction of the timings and the gather of the parity checksums.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]      # the CPU path timed on this box's host cores
    python bench.py --dump-outputs DIR ...                         # also write the last timed step's results (rank 0)

Prints ONE JSON line (rank 0).  Beyond the base contract it carries, all measured in the same run but OUTSIDE the
headline timed region:
  roofline      dominant kernel vs the measured HBM peak AND vs the integer roofline measured on this GPU
                (agx_measure_butterfly_peak: the butterfly instruction stream alone); `bound` names the lower one
  sustained     >= 2 s of back-to-back steps with >= 100 NVML samples (clock, power, throttle reasons)
  configs       BASELINE configs 3, 4 and the cfg-5 sizes (n = 1024, 2048), each with its own roofline
  strong        cfg 5's fixed 2^31/n global batch split over the ranks (n = 1024, 2048, 4096)
  parity_in_bench  FORWARD spectra of slices of every rank's shard against the oracle (global indices; shard sums
                gathered on rank 0), the all-ranks forward checksum, and the K-round-trip checksum
  cpu_baseline, e2e, clocks, gpu_launches, kernels
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "NTT+INTT/sec at n=4096, 30-bit q"
UNIT = "pairs/s"
N_DEFAULT = 4096
PRIMES = (1053818881, 1054015489, 1054212097)   # SEAL-Embedded 30-bit primes (SURVEY.md App. A)
PRIME = PRIMES[0]
BATCH_PER_GPU = 65536               # configs[1]
SEED = 1234                         # SURVEY.md s.8(d): timing seed
HBM_FALLBACK_GBS = 6650.0           # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
PARITY_HEAD, PARITY_TAIL = 3072, 1024   # polynomials of every shard whose forward spectra are compared with the oracle
DUMP_BYTES_PER_ARRAY = 16 << 20     # --dump-outputs: float64 data per file (both files with headers stay below 64 MB)


def host_threads() -> int:
    """All host threads this process may use -- not OMP_NUM_THREADS, which torchrun pins to 1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def make_config(n: int, B: int, world: int, strong_total: int = 0) -> dict:
    """The workload description -- identical for our arm and the reference arm."""
    return {"workload": f"configs[1]: n={n} single 30-bit prime q={PRIME}, batch of {B} polynomials per GPU, "
                        "forward NTT + inverse NTT over the batch, in place",
            "n": n, "nlimbs": 1, "batch_per_gpu": B, "global_batch": strong_total or world * B,
            "l2": f"inputs {B * n * 4 >> 20} MiB per GPU > 126 MB L2 (no flush needed)",
            "parallelism": f"batch-sharded x{world}, no collective"}


# ----------------------------------------------------------------------------------------------- clocks sampler

class ClockSampler:
    """Samples SM clock / power / throttle reasons of one GPU through NVML while a timed region runs."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, cuda_index: int, period_s: float = 0.002):
        self.samples, self.reasons, self.power = [], set(), []
        self.max_mhz = None
        self.period = period_s
        self._stop = threading.Event()
        self._thr = None
        self._h = None
        try:
            import pynvml
            import torch
            self._nv = pynvml
            pynvml.nvmlInit()
            h = None
            try:
                uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                idx = cuda_index
                if vis and all(v.strip().isdigit() for v in vis.split(",")):
                    idx = int(vis.split(",")[cuda_index])
                h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self._h = h
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # NVML missing: report that instead of inventing numbers
            self.error = repr(e)

    def _loop(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self._h) / 1000.0)
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        if self._h is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def stop(self) -> dict:
        self._stop.set()
        if self._thr:
            self._thr.join(2.0)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0,
                    "note": getattr(self, "error", "no samples")}
        return {"sm_mhz": int(statistics.median(self.samples)), "sm_mhz_min": min(self.samples),
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples),
                "power_w_max": round(max(self.power), 1) if self.power else None,
                "power_w_median": round(statistics.median(self.power), 1) if self.power else None}


# ------------------------------------------------------------------------------------------------ CPU baseline

def cpu_pairs_per_sec(n: int, primes, sample_polys: int, reps: int, variant: str, threads: int):
    """Time the oracle port (oracle/ntt_oracle.c) on `sample_polys` fwd+inv pairs, `reps` times; returns pairs/s."""
    from oracle import oracle as O
    P = O.Plan(n, primes)
    x = P.synthetic(sample_polys, seed=SEED)
    P.fwd(x, variant=variant, threads=threads)      # warm caches / thread pool
    P.inv(x, variant=variant, threads=threads)
    t0 = time.perf_counter()
    for _ in range(reps):
        P.fwd(x, variant=variant, threads=threads)
        P.inv(x, variant=variant, threads=threads)
    dt = time.perf_counter() - t0
    return sample_polys * len(primes) * reps / dt, dt


def reference_code_rate():
    """The reference's OWN kernel code (src/kernel/ntt.cpp compiled against the host SYCL stand-in, oracle/_ref), timed
    on the one BASELINE size it supports (n=1024, forward only, u64, one host thread -- it is a sequential emulation
    of the FPGA pipeline).  Returned as context next to the port's numbers; None where oracle/_ref was not built."""
    try:
        import numpy as np
        from oracle import oracle as O
        N, frames = 1024, 256
        if not O.ref_available(N):
            return None
        tw, pre = O.tables_u64(N, PRIME)
        x = (np.arange(N * frames, dtype=np.uint64) * np.uint64(2654435761)) % np.uint64(PRIME)
        O.reference_fwd_u64(N, x, x, PRIME, tw, pre, frames)
        t0 = time.perf_counter()
        reps = 4
        for _ in range(reps):
            O.reference_fwd_u64(N, x, x, PRIME, tw, pre, frames)
        dt = time.perf_counter() - t0
        return {"what": "reference's own fwd_ntt_kernel code via oracle/_ref, n=1024 forward u64, 1 thread",
                "forward_transforms_per_s": frames * reps / dt}
    except Exception as e:       # never let the context number break the bench line
        return {"error": repr(e)}


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's CPU implementation of the path, on this box's host cores.

    The reference's own kernel (src/kernel/ntt.cpp) is built only for N in {32,1024,8192,16384,32768} (ntt.h:11-23,
    #error otherwise), forward only, and needs the oneAPI FPGA emulator; n=4096 forward+inverse therefore runs the
    oracle port (oracle/ntt_oracle.c, Harvey/Shoup lazy butterflies = the arithmetic of ntt.cpp:331-393 at u32),
    OpenMP over polynomials on all host threads.  Same workload description as our arm; each STEP transforms a bounded
    sample of the 65,536-polynomial batch (the throughput is per pair, so the sample size does not enter the ratio)."""
    if rank != 0:
        return
    from oracle import oracle as O
    threads = host_threads()
    sample = min(args.cpu_sample, 16384)            # per step; K steps of this stay within a couple of minutes
    P = O.Plan(args.n, [PRIME])
    x = P.synthetic(sample, seed=SEED)
    for _ in range(max(1, min(args.warmup, 3))):
        P.fwd(x, threads=threads); P.inv(x, threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        P.fwd(x, threads=threads)
        P.inv(x, threads=threads)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": make_config(args.n, args.batch, max(world, args.gpus)),
        "sample_note": f"each step = bounded sample of {sample} of the {args.batch} polynomials (per-pair throughput)",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{sample} fwd+inv pairs per step x {args.steps} steps, Shoup-lazy C oracle, OpenMP",
                         "reference_code": reference_code_rate()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------- ours

def load_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(kernel_key: str):
    """DRAM bytes per launch from the ncu --set full capture of this build (profiles/roofline_traffic.json names the
    capture it was read from); None for kernels that were not captured."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        return d.get(kernel_key), d.get("_source")
    except Exception:
        return None, None


def dump_outputs(out_dir: str, ctx, data, B: int) -> None:
    """--dump-outputs: what the last timed step handed its caller, so that two builds can be compared output for output.
    A step is fwd then inv in place: its caller receives the forward spectra, then the batch back from the inverse.  Every
    step starts from the same batch (each is an exact round trip, checked by checksum), so the last step's spectra are
    recomputed here, after the timed region, from the batch it left behind, and the batch is restored.  A fixed, seeded
    sample of whole polynomials is written as float64 (exact for residues < 2^30): ntt_fwd.npy and ntt_inv.npy, both
    [rows][L][n]."""
    import numpy as np
    import torch
    L, n = ctx.L, ctx.n
    rows = max(1, min(B, DUMP_BYTES_PER_ARRAY // (L * n * 8)))
    idx = np.sort(np.random.default_rng(SEED).choice(B, size=rows, replace=False))
    sel = torch.from_numpy(idx).to(data.device)
    polys = data.view(B, L * n)

    def sample():
        return polys.index_select(0, sel).cpu().numpy().view(np.uint32).reshape(rows, L, n).astype(np.float64)

    inv_out = sample()
    ctx.fwd(data)
    fwd_out = sample()
    ctx.inv(data)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "ntt_fwd.npy"), fwd_out)
    np.save(os.path.join(out_dir, "ntt_inv.npy"), inv_out)


def run_ours(args, rank: int, local_rank: int, world: int):
    import numpy as np
    import torch
    import torch.distributed as dist
    import agilex_ntt_b200 as A

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference "
                         "for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # keep stdout to the one JSON line: NCCL prints its version banner on stdout when the communicator is
        # created, so point fd 1 at stderr while that happens
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def gather_u64(v: int):
        """Every rank's 64-bit value on every rank (as two 32-bit halves: no signed overflow anywhere)."""
        t = torch.tensor([v & 0xFFFFFFFF, v >> 32], dtype=torch.int64, device=dev)
        if world == 1:
            return [v]
        parts = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        return [int(p[0]) | (int(p[1]) << 32) for p in parts]

    stream = torch.cuda.current_stream()

    last_mhz = [None]

    def time_ms(fn, iters, warm=3):
        """Mean ms per call of fn (CUDA events on the launching stream), max over ranks; the SM clock NVML saw while the
        timed launches ran is left in last_mhz[0]."""
        for _ in range(warm):
            fn()
        barrier(); torch.cuda.synchronize()
        smp = ClockSampler(local_rank, period_s=0.001).start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(iters):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        last_mhz[0] = smp.stop().get("sm_mhz")
        barrier()
        return max_over_ranks([e0.elapsed_time(e1) / iters])[0]

    n, L, B = args.n, 1, args.batch
    if args.total_batch:                        # strong scaling (SURVEY.md s.8(d) cfg 5): a fixed global batch split over the ranks
        if args.total_batch % world:
            raise SystemExit("bench.py: --total-batch must be a multiple of the number of GPUs")
        B = args.total_batch // world
    ctx = A.Context(n, [PRIME], device=local_rank)
    data = torch.empty(B * L * n, dtype=torch.int32, device=dev)
    first_poly = rank * B
    ctx.fill_synthetic(data, seed=SEED, first_poly=first_poly)    # shard = slice of the global synthetic batch
    chk0 = ctx.checksum(data, first_index=first_poly * L * n)

    # ---- parity BEFORE timing: the forward spectra themselves (a wrong-but-invertible transform would survive a round
    # trip).  Head and tail slices of every rank's shard are checksummed with GLOBAL indices on the device, gathered,
    # and compared on rank 0 with the oracle's transform of the same global slices; the whole-shard forward checksum is
    # gathered too (reported, and compared with the oracle's whole batch when --full-parity).
    ctx.fwd(data)
    head, tail = min(PARITY_HEAD, B), min(PARITY_TAIL, B)
    slice_sum = (ctx.checksum(data[: head * n], first_index=first_poly * n)
                 + ctx.checksum(data[(B - tail) * n:], first_index=(first_poly + B - tail) * n)) % (1 << 64)
    fwd_sum = ctx.checksum(data, first_index=first_poly * n)
    slice_sums, fwd_sums = gather_u64(slice_sum), gather_u64(fwd_sum)
    ctx.inv(data)
    ok_roundtrip0 = ctx.checksum(data, first_index=first_poly * L * n) == chk0
    parity = {"forward_vs_oracle": None}
    if rank == 0:
        from oracle import oracle as O
        P = O.Plan(n, [PRIME])
        thr = host_threads()
        want = 0
        for r in range(world):
            for lo, cnt in ((r * B, head), (r * B + B - tail, tail)):
                y = P.fwd(P.synthetic(cnt, seed=SEED, first_poly=lo), threads=thr)
                want = (want + O.checksum_u32(y, first_index=lo * n)) % (1 << 64)
        got = A.combine_checksums(slice_sums)
        parity = {"forward_vs_oracle": "ok" if got == want else "FAILED",
                  "what": f"forward spectra of the first {head} and last {tail} polynomials of each of the {world} shards "
                          "(global indices), device checksums gathered over ranks == oracle's",
                  "forward_checksum_all_ranks": f"{A.combine_checksums(fwd_sums):016x}"}
        if args.full_parity:
            want_all = 0
            step = 8192
            for lo in range(0, world * B, step):
                y = P.fwd(P.synthetic(min(step, world * B - lo), seed=SEED, first_poly=lo), threads=thr)
                want_all = (want_all + O.checksum_u32(y, first_index=lo * n)) % (1 << 64)
            parity["forward_full_batch_vs_oracle"] = "ok" if want_all == A.combine_checksums(fwd_sums) else "FAILED"

    # ---- headline: W warm-up steps, then exactly K timed steps
    for _ in range(args.warmup):
        ctx.fwd(data); ctx.inv(data)
    torch.cuda.synchronize()

    K = args.steps
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    sampler = ClockSampler(local_rank)
    launches0 = ctx.launch_count()
    barrier(); torch.cuda.synchronize()
    sampler.start()
    t_wall0 = time.perf_counter()
    for k in range(K):
        ev[k][0].record(stream)
        ctx.fwd(data)
        ev[k][1].record(stream)
        ctx.inv(data)
        ev[k][2].record(stream)
    torch.cuda.synchronize(); barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    launches = ctx.launch_count() - launches0

    total_ms = ev[0][0].elapsed_time(ev[K - 1][2])
    fwd_ms = [ev[k][0].elapsed_time(ev[k][1]) for k in range(K)]
    inv_ms = [ev[k][1].elapsed_time(ev[k][2]) for k in range(K)]
    ok = ok_roundtrip0 and ctx.checksum(data, first_index=first_poly * L * n) == chk0   # K round trips leave the batch unchanged
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, data, B)
        ok = ok and ctx.checksum(data, first_index=first_poly * L * n) == chk0     # and so does the dump's extra one

    # ---- sustained: >= 2 s of back-to-back steps with NVML sampled throughout (a 20 ms burst says nothing about clocks)
    sustained = None
    if args.sustain_s > 0:
        per_step = total_ms / K
        reps = max(K, int(args.sustain_s * 1e3 / per_step) + 1)
        s_sampler = ClockSampler(local_rank, period_s=0.005)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        s_sampler.start()
        e0.record(stream)
        for _ in range(reps):
            ctx.fwd(data); ctx.inv(data)
        e1.record(stream)
        torch.cuda.synchronize(); barrier()
        s_clocks = s_sampler.stop()
        s_ms = max_over_ranks([e0.elapsed_time(e1)])[0]
        sustained = {"seconds": s_ms * 1e-3, "steps": reps, "value": world * B * L * reps / (s_ms * 1e-3), "unit": UNIT,
                     "ms_per_step": s_ms / reps, "clocks": s_clocks}
        ok = ok and ctx.checksum(data, first_index=first_poly * L * n) == chk0

    # ---- the integer roofline of THIS GPU: the butterfly instruction stream alone, 8 and 4 warps per scheduler
    bf_peak8, bf_mhz = ctx.measure_butterfly_peak(0, 1024)
    bf_peak4, _ = ctx.measure_butterfly_peak(0, 512)

    # ---- end-to-end through the host-pointer C ABI: pinned host buffers, H2D + kernels + D2H inside the timed region
    e2e_steps = max(1, min(K, args.e2e_steps))
    host = torch.empty(B * L * n, dtype=torch.int32).pin_memory()
    host.copy_(data)
    ctx.fwd_host(host)                                                     # warm the pipeline (allocations) ...
    ok_e2e_fwd = True
    if rank == 0:                                                          # ... and check a forward result of the host path
        from oracle import oracle as O
        P = O.Plan(n, [PRIME])
        yh = host[: 64 * n].numpy().view(np.uint32).reshape(64, 1, n)
        ok_e2e_fwd = bool((yh == P.fwd(P.synthetic(64, seed=SEED, first_poly=0), threads=4)).all())
    ctx.inv_host(host)
    barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ctx.fwd_host(host)      # returns once the spectra are back in host memory
        ctx.inv_host(host)
    torch.cuda.synchronize(); barrier()
    e2e_s = time.perf_counter() - t0
    ok_e2e = ok_e2e_fwd and bool((host[: 64 * n].to(dev) == data[: 64 * n]).all()) and \
        bool((host[-64 * n:].to(dev) == data[-64 * n:]).all())
    del host

    total_ms, e2e_ms, fwd_avg, inv_avg, bad = max_over_ranks(
        [total_ms, e2e_s * 1e3, statistics.mean(fwd_ms), statistics.mean(inv_ms), 0.0 if (ok and ok_e2e) else 1.0])

    peak, peak_src = load_peak()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count

    def roofline_of(kernel, nn, transforms, ms, bytes_per_unit, mhz, traffic_key=None, bf_per_transform=None):
        """One kernel (or fused op) against both rooflines: algorithmic bytes / measured HBM peak, and butterflies per
        clock per SM / the measured isolated-stream rate.  `bound` = whichever roofline allows fewer units per second."""
        logn = nn.bit_length() - 1
        byts = float(bytes_per_unit) * transforms
        achieved = byts / (ms * 1e-3) / 1e9
        bf = (nn // 2) * logn if bf_per_transform is None else bf_per_transform
        bf_rate = transforms * bf / (ms * 1e-3) / (sms * mhz * 1e6)
        hbm_units_s = peak * 1e9 / bytes_per_unit
        int_units_s = bf_peak8 * sms * mhz * 1e6 / bf
        traffic, tsrc = load_traffic(traffic_key) if traffic_key else (None, None)
        return {"bound": "hbm" if hbm_units_s <= int_units_s else "integer", "kernel": kernel, "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": tsrc,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": byts, "launch_ms": ms,
                "frac_of_8TBs": achieved / 8000.0,
                "integer": {"achieved": bf_rate, "peak": bf_peak8, "unit": "butterflies/clk/SM", "frac": bf_rate / bf_peak8,
                            "peak_4_warps_per_scheduler": bf_peak4, "peak_issue_limit_imad_hi_half_rate": 16.0,
                            "sm_mhz": mhz, "peak_source": "agx_measure_butterfly_peak on this GPU in this run "
                                                          f"(isolated butterfly stream, implied clock {bf_mhz:.0f} MHz)"},
                "roofline_units_per_s": {"hbm": hbm_units_s, "integer": int_units_s}}

    # ---- every other BASELINE config, device-resident, own buffers, same event method (outside the headline region)
    configs = {}
    if not args.no_extras:
        mhz_x = (sustained or {}).get("clocks", {}).get("sm_mhz") or clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965
        del data
        torch.cuda.empty_cache()

        def ntt_case(nn, LL, BB, key, what):
            c = A.Context(nn, PRIMES[:LL], device=local_rank)
            d = torch.empty(BB * LL * nn, dtype=torch.int32, device=dev)
            c.fill_synthetic(d, seed=SEED, first_poly=rank * BB)
            s0 = c.checksum(d, first_index=rank * BB * LL * nn)
            tf = time_ms(lambda: c.fwd(d), args.extra_iters)
            ti = time_ms(lambda: c.inv(d), args.extra_iters)
            mhz_c = last_mhz[0] or mhz_x
            c.fwd(d); c.inv(d)
            good = c.checksum(d, first_index=rank * BB * LL * nn) == s0
            T = BB * LL
            configs[key] = {"workload": what, "n": nn, "nlimbs": LL, "batch_per_gpu": BB,
                            "value": world * T / ((tf + ti) * 1e-3), "unit": "pairs/s",
                            "fwd_ms": tf, "inv_ms": ti, "variant": c.variant(), "round_trip": "ok" if good else "FAILED",
                            "roofline": roofline_of(("ntt_inv" if ti >= tf else "ntt_fwd") + f"<{c.variant()}>", nn, T,
                                                    max(tf, ti), 2 * nn * 4, mhz_c)}
            del d
            c.close()
            return good

        good = ntt_case(4096, 3, 32768, "cfg3", "configs[2]: n=4096, 3-limb RNS (SEAL-Embedded 30-bit primes), batch of 32,768")
        # cfg 4: negacyclic polynomial multiply n=2048, batch of 131,072: 3 n 4 B of algorithmic traffic per product
        nn, BB = 2048, 131072
        c = A.Context(nn, [PRIME], device=local_rank)
        a, b = (torch.empty(BB * nn, dtype=torch.int32, device=dev) for _ in range(2))
        out = torch.empty_like(a)
        c.fill_synthetic(a, seed=1, first_poly=rank * BB)
        c.fill_synthetic(b, seed=2, first_poly=rank * BB)
        l0 = c.launch_count()
        c.polymul(out, a, b)
        per_call = c.launch_count() - l0
        tp = time_ms(lambda: c.polymul(out, a, b), args.extra_iters)
        mhz_p = last_mhz[0] or mhz_x
        pm_ok = True
        if rank == 0:                    # exact schoolbook on a few products, NTT-path oracle on a slice
            from oracle import oracle as O
            P = O.Plan(nn, [PRIME])
            xa, xb = P.synthetic(256, seed=1), P.synthetic(256, seed=2)
            got = out[: 256 * nn].cpu().numpy().view(np.uint32).reshape(256, 1, nn)
            pm_ok = bool((got == P.polymul(xa, xb, threads=host_threads())).all())
            for i in (0, 255):
                pm_ok = pm_ok and bool((O.polymul_schoolbook(xa[i, 0], xb[i, 0], PRIME) == got[i, 0]).all())
        logn = 11
        configs["cfg4"] = {"workload": "configs[3]: negacyclic polynomial multiply n=2048 (NTT, pointwise modmul, INTT), batch of 131,072",
                           "n": nn, "nlimbs": 1, "batch_per_gpu": BB, "value": world * BB / (tp * 1e-3), "unit": "products/s",
                           "ms": tp, "launches_per_call": per_call, "vs_oracle_and_schoolbook": "ok" if pm_ok else "FAILED",
                           "roofline": roofline_of(f"polymul<n={nn}>, {per_call} launch(es)", nn, BB, tp, 3 * nn * 4, mhz_p,
                                                   bf_per_transform=3 * (nn // 2) * logn)}
        good = good and pm_ok
        # the same products with b kept in evaluation form (agx_polymul_by_spectrum: two launches, 5 streams of traffic):
        # SURVEY s.8(f) rank 4; must reproduce the three-launch product bit for bit
        want = c.checksum(out, first_index=rank * BB * nn)
        c.fwd(b)
        l0 = c.launch_count()
        c.polymul_by_spectrum(out, a, b)
        per_call_s = c.launch_count() - l0
        ps_ok = c.checksum(out, first_index=rank * BB * nn) == want
        ts = time_ms(lambda: c.polymul_by_spectrum(out, a, b), args.extra_iters)
        mhz_s = last_mhz[0] or mhz_x
        configs["cfg4_by_spectrum"] = {"workload": "configs[3] with one operand already transformed (c = INTT(NTT(a) .* b_hat)), n=2048, batch of 131,072",
                                       "n": nn, "nlimbs": 1, "batch_per_gpu": BB, "value": world * BB / (ts * 1e-3), "unit": "products/s",
                                       "ms": ts, "launches_per_call": per_call_s, "equals_agx_polymul": "ok" if ps_ok else "FAILED",
                                       "roofline": roofline_of(f"polymul_by_spectrum<n={nn}>, {per_call_s} launch(es)", nn, BB, ts,
                                                               3 * nn * 4, mhz_s, bf_per_transform=2 * (nn // 2) * logn)}
        good = good and ps_ok
        del a, b, out
        c.close()
        for nn in (1024, 2048):
            good = ntt_case(nn, 1, (1 << 28) // nn, f"cfg5_n{nn}",
                            f"configs[4] size n={nn}: single prime, 2^28/n = {(1 << 28) // nn} polynomials (1 GiB) per GPU") and good
        # strong scaling: cfg 5's fixed global batch of 2^31/n polynomials (8 GiB) split contiguously over the ranks
        strong = {}
        if not args.no_strong:
            for nn in (1024, 2048, 4096):
                total = (1 << 31) // nn
                BB = total // world
                c = A.Context(nn, [PRIME], device=local_rank)
                d = torch.empty(BB * nn, dtype=torch.int32, device=dev)
                c.fill_synthetic(d, seed=SEED, first_poly=rank * BB)
                s0 = c.checksum(d, first_index=rank * BB * nn)
                tf = time_ms(lambda: c.fwd(d), 5, warm=2)
                ti = time_ms(lambda: c.inv(d), 5, warm=2)
                c.fwd(d); c.inv(d)
                rt = c.checksum(d, first_index=rank * BB * nn) == s0
                good = good and rt
                strong[f"n{nn}"] = {"global_batch": total, "batch_per_gpu": BB, "fwd_ms": tf, "inv_ms": ti,
                                    "value": total / ((tf + ti) * 1e-3), "unit": "pairs/s", "scaling": "strong",
                                    "round_trip": "ok" if rt else "FAILED"}
                del d
                c.close()
        # the reference-shaped u64 path on device-resident frames (agx_ref_fwd_dev): N = 16384 (the reference's default,
        # main.cpp:9,27), a 60-bit NTT prime, 256 MiB of frames per GPU; fraction of the 2 N 8 B HBM roofline and of the
        # u64 integer roofline measured on this GPU (the ntt.cpp:331-369 butterfly stream alone)
        u64 = None
        try:
            N64, q64 = 16384, 1152921504606584833
            psi = next(c for c in (pow(g, (q64 - 1) // (2 * N64), q64) for g in range(2, 200)) if pow(c, N64, q64) == q64 - 1)
            pw = [1] * N64
            for i in range(1, N64):
                pw[i] = pw[i - 1] * psi % q64
            lg = N64.bit_length() - 1
            roots = [pw[int(format(k, f"0{lg}b")[::-1], 2)] for k in range(N64)]
            tw = np.array(roots, dtype=np.uint64)
            pre = np.array([(w << 64) // q64 for w in roots], dtype=np.uint64)
            frames = (256 << 20) // (N64 * 8)
            d_tw = torch.from_numpy(tw.view(np.int64)).to(dev)
            d_pre = torch.from_numpy(pre.view(np.int64)).to(dev)
            gen = torch.Generator(device=dev); gen.manual_seed(SEED + rank)
            d_in = torch.randint(0, 4 * q64, (frames * N64,), dtype=torch.int64, device=dev, generator=gen)   # lazy [0,4q)
            d_out = torch.empty_like(d_in)
            rp = A.RefPipeline(device=local_rank)
            rp.fwd_dev(N64, d_in, d_in, d_out, q64, d_tw, d_pre, frames)
            torch.cuda.synchronize()
            ok64 = True
            if rank == 0:
                from oracle import oracle as O
                xin = d_in[: 2 * N64].cpu().numpy().view(np.uint64)
                ok64 = bool((d_out[: 2 * N64].cpu().numpy().view(np.uint64) == O.ref_fwd_u64(xin, xin, q64, tw, pre, 2)).all())
            t64 = time_ms(lambda: rp.fwd_dev(N64, d_in, d_in, d_out, q64, d_tw, d_pre, frames), args.extra_iters)
            mhz_u = last_mhz[0] or mhz_x
            peak64, _ = ctx.measure_butterfly_peak(1, 1024)
            fps = world * frames / (t64 * 1e-3)
            bf64 = (N64 // 2) * lg
            rate = frames * bf64 / (t64 * 1e-3) / (sms * mhz_u * 1e6)
            hbm_fps, int_fps = peak * 1e9 / (2 * N64 * 8), peak64 * sms * mhz_u * 1e6 / bf64
            u64 = {"workload": f"reference-shaped u64 forward NTT (agx_ref_fwd_dev), N={N64}, 60-bit prime, {frames} frames per GPU, "
                               "lazy [0,4q) inputs, device resident",
                   "value": fps, "unit": "frames/s", "ms": t64, "vs_restatement": "ok" if ok64 else "FAILED",
                   "roofline": {"bound": "hbm" if hbm_fps <= int_fps else "integer", "achieved": frames * 2 * N64 * 8 / (t64 * 1e-3) / 1e9,
                                "peak": peak, "unit": "GB/s", "frac": frames * 2 * N64 * 8 / (t64 * 1e-3) / 1e9 / peak, "traffic": None,
                                "integer": {"achieved": rate, "peak": peak64, "unit": "u64 butterflies/clk/SM", "frac": rate / peak64,
                                            "sm_mhz": mhz_u},
                                "roofline_units_per_s": {"hbm": hbm_fps, "integer": int_fps}}}
            good = good and ok64
            del d_in, d_out
            rp.close()
        except Exception as e:       # a context number: never let it take the headline line down
            u64 = {"error": repr(e)}
        configs["u64_n16384"] = u64
        bad = max_over_ranks([bad, 0.0 if good else 1.0])[0]
    else:
        strong = {}

    if rank == 0:
        dom, dom_ms = ("ntt_fwd_kernel", fwd_avg) if fwd_avg >= inv_avg else ("ntt_inv_kernel", inv_avg)
        variant = ctx.variant()
        mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965
        bytes_per_launch = 2.0 * n * 4 * B * L                      # read once + write once (SURVEY.md s.8(d))
        roof = roofline_of(f"{dom}<{variant}>", n, B * L, dom_ms, 2 * n * 4, mhz, traffic_key=dom)
        failed = bad != 0.0 or parity.get("forward_vs_oracle") != "ok" or parity.get("forward_full_batch_vs_oracle") == "FAILED"
        parity["round_trips_and_e2e"] = "ok" if bad == 0.0 else "FAILED"
        line = {
            "metric": METRIC, "value": world * B * L * K / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": K, "warmup": args.warmup, "ms_per_step": total_ms / K, "higher_is_better": True,
            "scaling": "strong" if args.total_batch else "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": make_config(n, B, world, args.total_batch),
            "kernel_variant": variant,
            "roofline": roof,
            "kernels": {"ntt_fwd_ms": fwd_avg, "ntt_inv_ms": inv_avg,
                        "fwd_transforms_per_s": B * L / (fwd_avg * 1e-3), "inv_transforms_per_s": B * L / (inv_avg * 1e-3),
                        "fwd_GBps": bytes_per_launch / (fwd_avg * 1e-3) / 1e9,
                        "inv_GBps": bytes_per_launch / (inv_avg * 1e-3) / 1e9,
                        "fwd_frac_of_measured_hbm": bytes_per_launch / (fwd_avg * 1e-3) / 1e9 / peak,
                        "inv_frac_of_measured_hbm": bytes_per_launch / (inv_avg * 1e-3) / 1e9 / peak},
            "sustained": sustained,
            "e2e": {"value": world * B * L * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": 2 * B * L * n * 4, "d2h_bytes_per_step": 2 * B * L * n * 4,
                    "steps": e2e_steps, "api": "agx_ntt_fwd_host + agx_ntt_inv_host on pinned host buffers"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "configs": configs,
            "strong": strong,
            "parity_in_bench": parity,
            "wall_s_timed_region": t_wall,
        }
        if world == 1 and not args.no_cpu:
            thr = host_threads()
            sample = args.cpu_sample
            reps = 8                      # 262,144 pairs ~ 12 CPU-seconds of the Shoup-lazy port
            v, dt = cpu_pairs_per_sec(n, [PRIME], sample, reps, "shoup", thr)
            vb, _ = cpu_pairs_per_sec(n, [PRIME], sample, 1, "barrett", thr)
            v1, _ = cpu_pairs_per_sec(n, [PRIME], max(256, sample // 16), 1, "shoup", 1)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": thr, "kind": "port",
                                    "sample": f"{sample} of the {B} polynomials x {reps} reps, fwd+inv, Shoup-lazy C "
                                              f"oracle (ntt.cpp:331-393 arithmetic at u32), OpenMP x{thr}; "
                                              f"{dt:.1f} s wall",
                                    "barrett_value": vb, "single_core_value": v1,
                                    "reference_code": reference_code_rate()}
        print(json.dumps(line), flush=True)
        if failed:
            raise SystemExit("bench.py: parity check inside the bench FAILED: " + json.dumps(parity))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--n", "--ntt-size", dest="n", type=int, default=N_DEFAULT,
                    help="transform size (use --ntt-size under torchrun, whose own parser claims --n*)")
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="polynomials per GPU")
    ap.add_argument("--total-batch", type=int, default=0,
                    help="strong scaling: fixed global batch split contiguously over the GPUs (cfg 5 uses 2^31/n)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--sustain-s", type=float, default=2.2, help="length of the sustained block (0 = skip)")
    ap.add_argument("--extra-iters", type=int, default=20, help="timed launches per extra config")
    ap.add_argument("--cpu-sample", type=int, default=32768, help="polynomials in the bounded CPU sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip BASELINE configs 3-5 and the strong-scaling block")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--full-parity", action="store_true", help="also compare the whole forward batch with the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's results for a fixed sample of rank 0's polynomials: DIR/ntt_inv.npy "
                         "(the batch the last inverse returned) and DIR/ntt_fwd.npy (its forward spectra, recomputed "
                         "after the timed region from that batch by one more fwd + inv)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if world == 1 and args.gpus > 1 and args.impl == "ours":
        # launched without torchrun: re-exec under torch.distributed.run, one process per GPU
        import subprocess
        port = 29500 + os.getpid() % 2000
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
