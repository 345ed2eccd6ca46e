#!/usr/bin/env python
"""bench.py -- the BASELINE.json configurations on B200.

    python bench.py --gpus N --steps K --warmup W [--workload C2]   # this repo's CUDA path (default: C2, the headline)
    python bench.py --impl reference --gpus N --steps K ...          # the reference algorithm on the host cores
    python bench.py ... --dump-outputs DIR                           # also write a sample of the last step's result

Workloads (BASELINE.json `configs`, SURVEY.md section 8d):
  C1     PolyBenchmark forwardNtt, N=4096, one 55-bit modulus (Benchmarks/PolyBenchmark/PolyBenchmark.swift:148-158)
  C1-8192  the same at N=8192
  C2     Bfv<UInt64> ct x ct multiply, N=8192, 4 coefficient moduli, batch 1024 per GPU        <- the headline metric
  C2-L4  the same with 5 coefficient moduli (L=4)
  C2-u32 Bfv<UInt32> ct x ct multiply, N=4096, the 27/28/28-bit PIR default moduli (uint32 buffers end to end)
  C3     relinearize + modSwitchDown, N=16384, 8 coefficient moduli, batch 4096 sharded over the GPUs (strong scaling)
  C4     MulPir server computeResponse, 2^20 x 64 B index-PIR database, one shard per GPU (weak scaling)
  C5     PNNS CiphertextMatrix x plaintext-matrix, N=8192, 512-dimensional vectors, one row block per GPU

A "step" = one pass of the hot path over one batch of synthetic input.  `value` is device-resident throughput (inputs in
HBM before the clock starts, CUDA events on the launch stream, max over ranks); `e2e` is the same work through the
host-pointer C-ABI call with pinned host buffers (H2D + D2H inside the clock).  C4/C5 are host-API workloads (the
query arrives from the host every time): there `value` and `e2e` are the same measurement, and a step is one query on
each of the 8 concurrent host threads (C4) or one batch of 16 query vectors (C5).  Every timed loop runs --steps
iterations: the headline, `e2e` and the relinearize extras; only the roofline's lone-kernel timing is a fixed 20 launches.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "swift-homomorphic-encryption_b200")
for p in (ROOT, PKG, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

# Parameter sets (BASELINE.md section 3): the largest 55-bit NTT-friendly primes, descending -- what the reference's
# generatePrimes(significantBitCounts: [55,...], preferringSmall: false, nttDegree: N) returns (Scalar.swift:113-154);
# the first three at N=8192 are its predefined n_8192_logq_3x55 set (EncryptionParameters.swift:406-410); t = 557057
# is the 20-bit NTT-friendly plaintext modulus of RlweBenchmark (EncryptionParameters.swift:383).
Q4096 = [36028797018652673]
Q8192 = [36028797018652673, 36028797017571329, 36028797017456641, 36028797017276417, 36028797017014273]
Q16384 = [36028797017456641, 36028797016178689, 36028797014704129, 36028797014573057, 36028797014376449,
          36028797014081537, 36028797013327873, 36028797013098497]
WORKLOADS = {
    # name: (kind, N, coefficient moduli [q_0..q_{L-1}, q_ks], t, default batch)
    "C1": ("ntt", 4096, Q4096, 557057, 32768),
    "C1-8192": ("ntt", 8192, Q8192[:1], 557057, 16384),
    "C2": ("mul", 8192, Q8192[:4], 557057, 1024),
    "C2-L4": ("mul", 8192, Q8192[:5], 557057, 1024),
    "C3": ("relin", 16384, Q16384, 557057, 4096),
    # Bfv<UInt32> ct x ct multiply at the PIR default parameters n_4096_logq_27_28_28 (EncryptionParameters.swift:357-367)
    "C2-u32": ("mul32", 4096, [134176769, 268369921, 268361729], 17, 4096),
    "C4": ("pir", 4096, None, 17, 0),
    "C5": ("pnns", 8192, None, 65537, 0),
}
# Integer-multiply pipe ceiling of the 64-bit Shoup butterfly, measured with the butterfly alone in a loop
# (tools/mb_r2.cu under ncu, profiles/r02_microbench_pipes.txt): butterflies per clock per SM.
BUTTERFLY_PIPE_PEAK = {"value": 3.3, "unit": "butterflies/clk/SM",
                       "source": "profiles/r02_microbench_pipes.txt (Cooley-Tukey / Gentleman-Sande Shoup butterfly alone: "
                                 "3.2-3.4 at 4-16 warps per scheduler, multiply pipe 97-98 % busy)"}
DUMP_BYTES = 48 << 20  # size of the --dump-outputs sample (float32 limbs)


def workload_params(name):
    kind, n, moduli, t, batch = WORKLOADS[name]
    return n, list(moduli), t, batch


def stage_model_bytes(n, L):
    """Algorithmic bytes per multiply: SURVEY.md section 8(d) stage model (28R + 3L) N w."""
    R = 2 * L + 1
    return (28 * R + 3 * L) * n * 8


def relin_model_bytes(n, L):
    """SURVEY.md section 8(d): relinearize (2LK + 5L + 8K) N w plus modSwitchDown (4L - 2) N w at K = L + 1."""
    K = L + 1
    return ((2 * L * K + 5 * L + 8 * K) + (4 * L - 2)) * n * 8


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.rows = []
        self.idx = device_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.1] or [r for _, r in self.rows[-3:]]
        sm = sorted(int(float(r[1])) for r in rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in rows:
            for k, name in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(rows)}


def host_threads():
    """All host threads this process may use (torchrun pins OMP_NUM_THREADS=1, which is not what we want here)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_quota():
    """CPU bandwidth limit of this container in cores (cgroup v2 cpu.max), or None when unlimited / unknown."""
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if quota == "max" else max(1, -(-int(quota) // int(period)))
    except Exception:
        return None


# ====================================================================================== CPU arm (the oracle port)
def cpu_items(kind, ctx, n, L, count, seed):
    """Synthetic inputs of `count` units for the oracle."""
    from oracle import oracle as orc

    if kind in ("mul", "mul32"):
        return (orc.fill_uniform(seed, ctx.q, n, count * 2 * L).reshape(count, 2, L, n),
                orc.fill_uniform(seed + 1, ctx.q, n, count * 2 * L).reshape(count, 2, L, n))
    if kind == "relin":
        return (orc.fill_uniform(seed, ctx.q, n, count * 3 * L).reshape(count, 3, L, n),)
    return (orc.fill_uniform(seed, ctx.q[:1], n, count).reshape(count, 1, n),)


def cpu_run(kind, ctx, items, threads, relin_key=None):
    from oracle import oracle as orc

    if kind in ("mul", "mul32"):
        return ctx.mul(items[0], items[1], threads=threads)
    if kind == "relin":
        return ctx.mod_switch_down(ctx.relinearize(items[0], relin_key, threads=threads), threads=threads)
    return orc.ntt_forward_inplace(ctx.n, ctx.q[:1], items[0], threads)  # in place, OpenMP over rows


def best_thread_count(kind, ctx, n, L, relin_key):
    """All logical CPUs, half of them (one per physical core) or the container's CPU quota, whichever runs the oracle
    fastest on a short probe -- the CPU baseline should get its best configuration."""
    full = host_threads()
    if kind == "ntt":
        return full
    candidates = {full, max(1, full // 2)}
    if cpu_quota():
        candidates.add(min(full, cpu_quota()))
    best, best_rate = full, 0.0
    for c in sorted(candidates, reverse=True):
        k = 2 * c
        items = cpu_items(kind, ctx, n, L, k, 11)
        cpu_run(kind, ctx, tuple(x[:c] for x in items), c, relin_key)  # warm the threads / page in
        t0 = time.perf_counter()
        cpu_run(kind, ctx, items, c, relin_key)
        rate = k / (time.perf_counter() - t0)
        if rate > best_rate:
            best, best_rate = c, rate
    return best


def cpu_context(kind, n, moduli, t):
    from oracle import oracle as orc

    if len(moduli) == 1:  # the oracle's context wants a key-switching modulus; the NTT arm never touches it
        moduli = list(moduli) + [p for p in orc.generate_primes([55, 55], False, n) if p != moduli[0]][:1]
    ctx = orc.Context(n, moduli, t, word_bits=32 if kind == "mul32" else 64)
    relin_key = ctx.keygen(5)[1] if kind == "relin" else None
    return ctx, relin_key


def cpu_reference_throughput(kind, n, moduli, t, budget_s=12.0):
    """Times the oracle (C restatement of the Swift reference) on a bounded sample of the same workload."""
    ctx, relin_key = cpu_context(kind, n, moduli, t)
    L = ctx.L
    cores = best_thread_count(kind, ctx, n, L, relin_key)
    probe = max(1, min(cores, 8)) * (64 if kind == "ntt" else 1)
    items = cpu_items(kind, ctx, n, L, probe, 1)
    t0 = time.perf_counter()
    cpu_run(kind, ctx, items, cores, relin_key)
    per_round = time.perf_counter() - t0
    sample = int(max(cores, min(1 << 16 if kind == "ntt" else 4096, budget_s / max(per_round, 1e-4) * probe)))
    sample = (sample // cores) * cores or cores
    items = cpu_items(kind, ctx, n, L, sample, 3)
    t0 = time.perf_counter()
    cpu_run(kind, ctx, items, cores, relin_key)
    dt = time.perf_counter() - t0
    return sample / dt, cores, sample, dt


METRICS = {
    "ntt": ("forward NTT/s (PolyRq.forwardNtt), one 55-bit modulus", "NTT/s"),
    "mul": ("BFV ct*ct mults/sec at N=8192, 4 coefficient moduli", "mult/s"),
    "mul32": ("Bfv<UInt32> ct*ct mults/sec at N=4096, 27/28/28-bit coefficient moduli", "mult/s"),
    "relin": ("Bfv relinearize + modSwitchDown per second at N=16384, 8 coefficient moduli", "ciphertexts/s"),
    "pir": ("MulPir computeResponse queries/s (index PIR, 2^20 x 64 B database resident in HBM)", "queries/s"),
    "pnns": ("PNNS encrypted dot products/s (mulTranspose + modSwitchDownToSingle, 512-dimensional vectors)", "dot products/s"),
}


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; no Swift toolchain here) on all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind = WORKLOADS[args.workload][0]
    metric, unit = METRICS[kind]
    base = {"impl": "reference", "metric": metric, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "vs_baseline": None, "dtype": "u32" if kind == "mul32" else "u64",
            "data": "synthetic",
            "scaling": "strong" if kind == "relin" else "weak"}
    if kind in ("pir", "pnns"):
        # the application drivers' CPU arm is the oracle timed on a bounded slice of one query, scaled (tools/bench_*.py)
        print(json.dumps({**base, "unavailable": "the CPU restatement of this application driver is timed beside the GPU "
                                                 "arm on a bounded slice (cpu_baseline in the b200 line); it has no standalone arm"}))
        return
    n, moduli, t, _ = workload_params(args.workload)
    ctx, relin_key = cpu_context(kind, n, moduli, t)
    L = ctx.L
    cores = best_thread_count(kind, ctx, n, L, relin_key)
    sample = max(cores, 2 * cores) * (256 if kind == "ntt" else 1)  # bounded per-step sample of the batch
    items = cpu_items(kind, ctx, n, L, sample, 3)
    for _ in range(args.warmup):
        cpu_run(kind, ctx, items, cores, relin_key)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_run(kind, ctx, items, cores, relin_key)
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {**base, "value": value, "ms_per_step": dt / args.steps * 1e3,
            "config": {"workload": f"{args.workload}: N={n}, {len(moduli)} coefficient moduli (L={L}), CPU sample of {sample} "
                                   f"units per step"},
            "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": "port", "cpu_quota_cores": cpu_quota(),
                             "sample": f"{sample} units/step x {args.steps} steps, OpenMP over units, C restatement of the "
                                       "Swift reference (no Swift toolchain on this box)"},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ====================================================================================== GPU arm
class Harness:
    """Process group, clocks and the timed loop shared by the device-resident workloads."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        import hecuda

        self.torch, self.dist, self.hecuda = torch, dist, hecuda
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available() or hecuda.device_count() < 1:
            raise SystemExit("bench.py needs a CUDA device (the product has no CPU fallback)")
        torch.cuda.set_device(self.local_rank)
        hecuda.set_device(self.local_rank)
        self.affinity0 = os.sched_getaffinity(0)
        try:  # host threads and pinned staging next to the GPU (NUMA node of its PCIe root)
            self.numa = hecuda.bind_host_to_device(self.local_rank)
        except Exception as exc:  # noqa: BLE001
            self.numa = {"error": repr(exc)}
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.dev = torch.device("cuda", self.local_rank)
        self.lib = hecuda.load_library()
        self.args = args
        self.stream = torch.cuda.current_stream()
        self.gen = torch.Generator(device=self.dev)
        self.gen.manual_seed(1234 + self.rank)

    def uniform(self, shape, moduli):
        """Uniform residues in [0, q_i) along the second-to-last axis (valid ring elements; SURVEY.md 8(d) flavour i)."""
        torch = self.torch
        qs = torch.tensor(list(moduli), dtype=torch.int64, device=self.dev).view(*([1] * (len(shape) - 2)), len(moduli), 1)
        x = torch.randint(0, 1 << 62, shape, generator=self.gen, device=self.dev, dtype=torch.int64)
        return (x % qs).contiguous()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def check(self, rc):
        if rc != 0:
            raise RuntimeError(self.lib.hecuda_last_error().decode())

    def timed(self, step, steps, warmup, sample_clocks=True):
        """W warm-up steps, then exactly K steps between barrier + synchronize, CUDA events on the launch stream, max
        over ranks.  Returns (total ms, kernel launches, clocks)."""
        torch = self.torch
        for _ in range(warmup):
            step()
        self.barrier()
        sampler = ClockSampler(self.local_rank) if (sample_clocks and self.rank == 0) else None
        if sampler:
            sampler.start()
            time.sleep(0.25)
        launches0 = self.hecuda.kernel_launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        w0 = time.perf_counter()
        ev0.record(self.stream)
        for _ in range(steps):
            step()
        ev1.record(self.stream)
        self.barrier()
        w1 = time.perf_counter()
        ms = self.max_over_ranks(ev0.elapsed_time(ev1))
        launches = self.hecuda.kernel_launch_count() - launches0
        clocks = sampler.stop(w0, w1) if sampler else None
        return ms, int(launches), clocks

    def kernel_time_ms(self, fn, reps=20, warm=3):
        torch = self.torch
        for _ in range(warm):
            fn()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        k0.record(self.stream)
        for _ in range(reps):
            fn()
        k1.record(self.stream)
        torch.cuda.synchronize()
        return k0.elapsed_time(k1) / reps

    def dump(self, name, result):
        """--dump-outputs DIR: a fixed, seeded sample of the units (first axis) of `result` as DIR/<name>.npy, rank 0 only.
        Residues reach 62 bits and float64 holds 53 exactly, so each residue is written as its four 16-bit limbs (least
        significant first, a trailing axis of 4) in float32: exact, and a change in any bit of a residue shows as a
        difference of at least 1."""
        out_dir = self.args.dump_outputs
        if not out_dir or self.rank != 0:
            return
        count = min(result.shape[0], max(1, DUMP_BYTES // (result[0].numel() * 4 * 4)))
        idx = np.sort(np.random.default_rng(0).choice(result.shape[0], count, replace=False))
        sample = result[self.torch.from_numpy(idx).to(result.device)].cpu().numpy().view(np.uint64)
        limbs = (sample[..., None] >> np.arange(0, 64, 16, dtype=np.uint64)) & np.uint64(0xFFFF)
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, f"{name}.npy"), limbs.astype(np.float32))

    def finish(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def ntt_roofline(h, ctx, base, rows_per_poly, polys, n, label, traffic_key=None):
    """The NTT kernel timed alone: HBM fraction (algorithmic 2 N w bytes per row) and fraction of the measured
    integer-multiply-pipe ceiling of its butterflies."""
    peak, peak_src = hbm_peak()
    buf = h.torch.randint(0, 1 << 50, (polys, rows_per_poly, n), device=h.dev, dtype=h.torch.int64)
    ms = h.kernel_time_ms(lambda: h.check(h.lib.hecuda_ntt_forward_device(ctx._h, base, buf.data_ptr(), rows_per_poly, polys,
                                                                       h.stream.cuda_stream)))
    rows = polys * rows_per_poly
    nbytes = rows * 2 * n * 8
    gbs = nbytes / (ms / 1e3) / 1e9
    logn = n.bit_length() - 1
    butterflies = rows * (n // 2) * logn
    sm_count = h.torch.cuda.get_device_properties(h.dev).multi_processor_count
    sm_mhz = 1965.0
    try:
        sm_mhz = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["sm_max_mhz"])
    except Exception:
        pass
    bfly_rate = butterflies / (ms / 1e3) / (sm_count * sm_mhz * 1e6)
    traffic = None
    tr_path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if traffic_key and os.path.exists(tr_path):
        tr = json.load(open(tr_path))
        if traffic_key in tr:  # per-row DRAM bytes of this kernel from the ncu --set full capture
            traffic = tr[traffic_key] * rows
    del buf
    return {"bound": "int_pipe", "kernel": label, "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
            "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": nbytes, "rows_per_launch": rows,
            "ntt_per_s": rows / (ms / 1e3), "launch_ms": ms,
            "bounds": {
                "hbm": {"achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak},
                "int_pipe": {"achieved": bfly_rate, "peak": BUTTERFLY_PIPE_PEAK["value"], "unit": BUTTERFLY_PIPE_PEAK["unit"],
                             "frac": bfly_rate / BUTTERFLY_PIPE_PEAK["value"], "peak_source": BUTTERFLY_PIPE_PEAK["source"],
                             "at_sm_mhz": sm_mhz},
                "binding": "int_pipe: the 64-bit Shoup butterflies keep the integer-multiply pipe (IMAD.WIDE 4 cycles, IMAD 2 "
                           "cycles per warp) busy while DRAM sits near 25 %; top-level achieved/peak/frac are the HBM figures"}}


def run_ntt(h, name):
    """C1: PolyBenchmark forwardNtt -- rows of one 55-bit modulus, in place."""
    args, hecuda = h.args, h.hecuda
    n, moduli, t, batch = workload_params(name)
    batch = args.batch or batch
    ctx = hecuda.Context(n, moduli, t)
    data = h.uniform((batch, 1, n), moduli[:1])

    def step():
        h.check(h.lib.hecuda_ntt_forward_device(ctx._h, hecuda.BASE_Q, data.data_ptr(), 1, batch, h.stream.cuda_stream))

    ms, launches, clocks = h.timed(step, args.steps, args.warmup)
    h.dump("ntt", data)
    value = h.world * batch * args.steps / (ms / 1e3)
    roofline = ntt_roofline(h, ctx, hecuda.BASE_Q, 1, batch, n, f"ntt_rows_kernel<{n.bit_length() - 1}, forward> (one NARROW modulus)")
    e2e = None
    if not args.no_e2e:
        hb = hecuda.PinnedBuffer((batch, 1, n))
        hb.array[...] = data.cpu().numpy().view(np.uint64)
        steps = args.steps
        h.check(h.lib.hecuda_ntt_forward(ctx._h, hecuda.BASE_Q, hb.array.ctypes.data, 1, batch))
        h.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            h.check(h.lib.hecuda_ntt_forward(ctx._h, hecuda.BASE_Q, hb.array.ctypes.data, 1, batch))
        dt = h.max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": h.world * batch * steps / dt, "unit": "NTT/s", "h2d_bytes_per_step": int(hb.array.nbytes),
               "d2h_bytes_per_step": int(hb.array.nbytes), "steps": steps,
               "timer": "host wall clock around blocking C-ABI calls (in-place transform of pinned host rows), max over ranks"}
        hb.free()
    config = {"workload": f"{name}: PolyRq.forwardNtt N={n}, one 55-bit modulus, {batch} rows per GPU per step, in place",
              "batch_per_gpu": batch, "parallelism": f"row-sharded x{h.world}, no data-path collective",
              "l2": f"rows per step ({batch * n * 8 / 1e6:.0f} MB) exceed L2 (126 MB); no explicit flush"}
    return dict(kind="ntt", n=n, moduli=moduli, t=t, value=value, ms=ms, launches=launches, clocks=clocks, roofline=roofline,
                e2e=e2e, config=config, scaling="weak", extra={})


def oracle_sample_check(kind, n, moduli, t, inputs, got, relin_key=None):
    """Outside the timed region: a sample of the device results against the oracle (bit-exact)."""
    try:
        from oracle import oracle as orc

        o = orc.Context(n, moduli, t, word_bits=32 if kind == "mul32" else 64)
        if kind in ("mul", "mul32"):
            want = o.mul(inputs[0], inputs[1])
        else:
            want = o.mod_switch_down(o.relinearize(inputs[0], relin_key))
        return bool(np.array_equal(want, got))
    except Exception as exc:  # noqa: BLE001
        return f"not checked: {exc!r}"


def run_mul(h, name):
    """C2: Bfv.mulAssign over a batch of synthetic ciphertext pairs.  C2-u32: the same for a Bfv<UInt32> context -- the
    device-resident value uses the residues zero-extended in 64-bit slots (how they live in HBM), the end-to-end value
    the uint32 entry point (4-byte residues across PCIe)."""
    args, hecuda, torch = h.args, h.hecuda, h.torch
    n, moduli, t, batch = workload_params(name)
    batch = args.batch or batch
    word32 = WORKLOADS[name][0] == "mul32"
    kind = "mul32" if word32 else "mul"
    ctx = hecuda.Context(n, moduli, t, scalar=np.uint32 if word32 else np.uint64)
    L = ctx.L
    lhs, rhs = h.uniform((batch, 2, L, n), moduli[:L]), h.uniform((batch, 2, L, n), moduli[:L])
    out = torch.empty((batch, 3, L, n), dtype=torch.int64, device=h.dev)

    def step():
        h.check(h.lib.hecuda_bfv_multiply_device(ctx._h, lhs.data_ptr(), rhs.data_ptr(), out.data_ptr(), batch,
                                                 h.stream.cuda_stream))

    ms, launches, clocks = h.timed(step, args.steps, args.warmup)
    h.dump("product", out)
    value = h.world * batch * args.steps / (ms / 1e3)
    peak, _ = hbm_peak()
    R = 2 * L + 1
    # the dominant kernel: forward NTT over the extended base the multiply computes in (28 of its 49 NTTs), timed
    # alone at the launch shape it has inside the timed step (the device path works in chunks of ~2 GB of scratch:
    # capi.cu, hecuda_context_create)
    device_chunk = max(1, min(4096, (2048 * 1024 * 1024) // (7 * R * n * 8)))
    roofline = ntt_roofline(h, ctx, hecuda.BASE_Q_AUX, R, min(batch, device_chunk) * 4, n,
                            f"ntt_rows_kernel<{n.bit_length() - 1}, forward> over [Q, aux] ({R} "
                            f"{'SMALL (32-bit butterfly)' if word32 else 'NARROW'} rows per polynomial)",
                            None if word32 else "ntt_forward_dram_bytes_per_row_narrow")
    if word32:
        roofline["bounds"]["int_pipe"]["note"] = ("the 3.3 butterflies/clk/SM ceiling is the 64-bit butterfly's; the 32-bit butterfly "
                                                  "(1 IMAD.HI + 2 IMAD) is ~3.5x cheaper, so this kernel leans on shared memory / issue")
    roofline["whole_step_stage_model"] = {
        "bytes_per_mult": stage_model_bytes(n, L), "achieved_gbs": stage_model_bytes(n, L) * (value / h.world) / 1e9,
        "frac": stage_model_bytes(n, L) * (value / h.world) / 1e9 / peak}
    checked = 4
    sample_ok = oracle_sample_check(kind, n, moduli, t, (lhs[:checked].cpu().numpy().view(np.uint64),
                                                           rhs[:checked].cpu().numpy().view(np.uint64)),
                                    out[:checked].cpu().numpy().view(np.uint64)) if h.rank == 0 else None

    # ---- extra (not the headline): relinearize and multiply+relinearize on the same batch.  The relinearization
    # key is synthetic (uniform residues, valid Eval-format rows): rank 0 creates it and it reaches the other ranks
    # by one NCCL broadcast into their key buffers (the only collective of the deployment, SURVEY.md 8e).
    extra = {"device_result_matches_oracle": {"pairs_checked": checked, "ok": sample_ok}}
    try:
        from hecuda import distributed as hd

        K = L + 1
        if h.rank == 0:
            key_host = h.uniform((L, 2, K, n), moduli).cpu().numpy().view(np.uint64)
        else:
            key_host = None
        evk = hd.broadcast_evaluation_key(ctx, key_host, src=0)
        relin_out = torch.empty((batch, 2, L, n), dtype=torch.int64, device=h.dev)

        def relin_step():
            h.check(h.lib.hecuda_bfv_relinearize_device(ctx._h, evk._h, out.data_ptr(), L, relin_out.data_ptr(), batch,
                                                        h.stream.cuda_stream))

        reps = args.steps
        for label, fn in (("relinearize_per_s", relin_step), ("multiply_relinearize_per_s", lambda: (step(), relin_step()))):
            tt, _, _ = h.timed(fn, reps, 2, sample_clocks=False)
            extra[label] = h.world * batch * reps / (tt / 1e3)
        extra["key_broadcast"] = "nccl" if h.world > 1 else "local"
        evk.close()
        del relin_out
    except Exception as exc:  # the headline number must survive a failure of the extras
        extra["error"] = repr(exc)

    # ---- e2e: host buffers (pinned), H2D + D2H inside the timed region, through the host-pointer C-ABI call
    e2e = None
    if not args.no_e2e:
        dt_host = np.uint32 if word32 else np.uint64
        hl, hr = hecuda.PinnedBuffer((batch, 2, L, n), dt_host), hecuda.PinnedBuffer((batch, 2, L, n), dt_host)
        ho = hecuda.PinnedBuffer((batch, 3, L, n), dt_host)
        hl.array[...] = lhs.cpu().numpy().view(np.uint64)
        hr.array[...] = rhs.cpu().numpy().view(np.uint64)
        steps = args.steps

        def host_mul():
            if word32:
                h.check(h.lib.hecuda_u32_bfv_multiply(ctx._h, hl.array.ctypes.data, hr.array.ctypes.data, ho.array.ctypes.data, batch))
            else:
                hecuda.Bfv.mulAssign(ctx, hl.array, hr.array, out=ho.array)

        host_mul()  # warm-up
        h.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            host_mul()
        torch.cuda.synchronize()
        dt = h.max_over_ranks(time.perf_counter() - t0)
        if not word32 and "error" not in extra and h.world == 1:
            # the fused call a server would make: multiply + relinearize + modSwitchDown, only 2 x (L-1) rows come back
            try:
                kh = h.uniform((L, 2, L + 1, n), moduli).cpu().numpy().view(np.uint64)
                evk2 = hecuda.EvaluationKey(ctx, kh)
                hf = hecuda.PinnedBuffer((batch, 2, L - 1, n))
                hecuda.Bfv.mulRelinearize(ctx, hl.array, hr.array, evk2, modSwitchDown=True, out=hf.array)
                f0 = time.perf_counter()
                for _ in range(steps):
                    hecuda.Bfv.mulRelinearize(ctx, hl.array, hr.array, evk2, modSwitchDown=True, out=hf.array)
                fdt = time.perf_counter() - f0
                extra["e2e_multiply_relinearize_modswitch"] = {
                    "value": batch * steps / fdt, "unit": "ciphertexts/s", "h2d_bytes_per_step": int(hl.array.nbytes + hr.array.nbytes),
                    "d2h_bytes_per_step": int(hf.array.nbytes), "call": "hecuda_bfv_multiply_relinearize(mod_switch = 1)"}
                hf.free()
                evk2.close()
            except Exception as exc:  # noqa: BLE001
                extra["e2e_multiply_relinearize_modswitch"] = {"error": repr(exc)}
        e2e = {"value": h.world * batch * steps / dt, "unit": "mult/s",
               "h2d_bytes_per_step": int(hl.array.nbytes + hr.array.nbytes), "d2h_bytes_per_step": int(ho.array.nbytes),
               "steps": steps, "timer": "host wall clock around blocking C-ABI calls, max over ranks",
               "matches_device_result": bool(np.array_equal(ho.array[:2], out[:2].cpu().numpy().view(np.uint64))),
               "host_numa": h.numa}
        hl.free(), hr.free(), ho.free()
    config = {"workload": f"{name}: Bfv<{'UInt32' if word32 else 'UInt64'}> ct*ct multiply (Bfv.mulAssign) N={n}, {len(moduli)} "
                          f"coefficient moduli (L={L} ciphertext + key-switch), t={t}, batch={batch} pairs per GPU",
              "batch_per_gpu": batch, "parallelism": f"batch-sharded x{h.world}, no data-path collective",
              "l2": f"inputs+outputs per step ({(lhs.numel() * 2 + out.numel()) * 8 / 1e9:.1f} GB) exceed L2 (126 MB); no explicit flush",
              "auxiliary_base": (f"L+1 primes below 2^{max(ctx.auxModuli).bit_length()} (BASE_Q_AUX)"
                                 if ctx.auxModuli != ctx.bskModuli else "reference Bsk"),
              "pipeline_chunk": int(os.environ.get("HECUDA_CHUNK", "0")) or "auto"}
    return dict(kind=kind, n=n, moduli=moduli, t=t, value=value, ms=ms, launches=launches, clocks=clocks, roofline=roofline,
                e2e=e2e, config=config, scaling="weak", extra=extra)


def run_relin(h, name):
    """C3: Bfv.relinearize + Bfv.modSwitchDown, batch sharded over the GPUs (strong scaling: the batch is fixed)."""
    args, hecuda, torch = h.args, h.hecuda, h.torch
    from hecuda import distributed as hd

    n, moduli, t, batch = workload_params(name)
    total = args.batch or batch
    lo, hi = hd.shard_range(total, h.rank, h.world)
    mine = hi - lo
    ctx = hecuda.Context(n, moduli, t)
    L, K = ctx.L, ctx.L + 1
    ct3 = h.uniform((mine, 3, L, n), moduli[:L])
    key_host = h.uniform((L, 2, K, n), moduli).cpu().numpy().view(np.uint64) if h.rank == 0 else None
    evk = hd.broadcast_evaluation_key(ctx, key_host, src=0)
    relin = torch.empty((mine, 2, L, n), dtype=torch.int64, device=h.dev)
    down = torch.empty((mine, 2, L - 1, n), dtype=torch.int64, device=h.dev)

    def step():
        h.check(h.lib.hecuda_bfv_relinearize_device(ctx._h, evk._h, ct3.data_ptr(), L, relin.data_ptr(), mine, h.stream.cuda_stream))
        h.check(h.lib.hecuda_bfv_mod_switch_down_device(ctx._h, relin.data_ptr(), 2, L, down.data_ptr(), mine, h.stream.cuda_stream))

    ms, launches, clocks = h.timed(step, args.steps, args.warmup)
    h.dump("mod_switched", down)
    value = total * args.steps / (ms / 1e3)
    peak, _ = hbm_peak()
    roofline = ntt_roofline(h, ctx, hecuda.BASE_KEYSWITCH, K, min(mine, 256), n,
                            "ntt_rows_kernel<14, forward> over [Q, q_ks] (the key-switch digit rows use the same kernel)")
    roofline["whole_step_stage_model"] = {
        "bytes_per_unit": relin_model_bytes(n, L), "achieved_gbs": relin_model_bytes(n, L) * (value / h.world) / 1e9,
        "frac": relin_model_bytes(n, L) * (value / h.world) / 1e9 / peak}
    sample_ok = None
    if h.rank == 0:
        sample_ok = oracle_sample_check("relin", n, moduli, t, (ct3[:2].cpu().numpy().view(np.uint64),),
                                        down[:2].cpu().numpy().view(np.uint64), relin_key=key_host)
    extra = {"device_result_matches_oracle": {"ciphertexts_checked": 2, "ok": sample_ok},
             "key_broadcast": "nccl" if h.world > 1 else "local"}
    e2e = None
    if not args.no_e2e:
        eb = min(mine, 512)
        hin, hmid = hecuda.PinnedBuffer((eb, 3, L, n)), hecuda.PinnedBuffer((eb, 2, L, n))
        hout = hecuda.PinnedBuffer((eb, 2, L - 1, n))
        hin.array[...] = ct3[:eb].cpu().numpy().view(np.uint64)
        steps = args.steps

        def host_step():
            hecuda.Bfv.relinearize(ctx, hin.array, evk, out=hmid.array)
            hecuda.Bfv.modSwitchDown(ctx, hmid.array, out=hout.array)

        host_step()
        h.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            host_step()
        dt = h.max_over_ranks(time.perf_counter() - t0)
        two_calls = {"value": h.world * eb * steps / dt, "unit": "ciphertexts/s",
                     "h2d_bytes_per_step": int(hin.array.nbytes + hmid.array.nbytes),
                     "d2h_bytes_per_step": int(hmid.array.nbytes + hout.array.nbytes),
                     "calls": "hecuda_bfv_relinearize then hecuda_bfv_mod_switch_down (the intermediate ciphertext crosses PCIe twice)"}
        extra["e2e_two_calls"] = two_calls
        # the same two operations as ONE public call: the relinearized ciphertext never leaves the device
        hecuda.Bfv.relinearizeModSwitchDown(ctx, hin.array, evk, out=hout.array)
        h.barrier()
        f0 = time.perf_counter()
        for _ in range(steps):
            hecuda.Bfv.relinearizeModSwitchDown(ctx, hin.array, evk, out=hout.array)
        fdt = h.max_over_ranks(time.perf_counter() - f0)
        e2e = {"value": h.world * eb * steps / fdt, "unit": "ciphertexts/s",
               "h2d_bytes_per_step": int(hin.array.nbytes), "d2h_bytes_per_step": int(hout.array.nbytes), "steps": steps,
               "batch_per_gpu": eb, "call": "hecuda_bfv_relinearize_mod_switch_down (relinearize + modSwitchDown in one pass)",
               "timer": "host wall clock around the blocking C-ABI call, max over ranks",
               "matches_device_result": bool(np.array_equal(hout.array[:2], down[:2].cpu().numpy().view(np.uint64)))}
        hin.free(), hmid.free(), hout.free()
    evk.close()
    config = {"workload": f"{name}: Bfv.relinearize + Bfv.modSwitchDown N={n}, {len(moduli)} coefficient moduli (L={L}), "
                          f"batch={total} ciphertexts sharded over {h.world} GPU(s)",
              "global_batch": total, "batch_per_gpu": mine, "parallelism": f"batch-sharded x{h.world}, key broadcast once (NCCL)",
              "l2": f"inputs+outputs per step ({(ct3.numel() + relin.numel() + down.numel()) * 8 / 1e9:.1f} GB) exceed L2; no explicit flush"}
    return dict(kind="relin", n=n, moduli=moduli, t=t, value=value, ms=ms, launches=launches, clocks=clocks,
                roofline=roofline, e2e=e2e, config=config, scaling="strong", extra=extra)


def run_app(args, name):
    """C4 / C5: the application drivers (tools/bench_pir.py, tools/bench_pnns.py) through the host-pointer API."""
    import hecuda

    kind = WORKLOADS[name][0]
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    hecuda.set_device(local_rank)
    try:
        numa = hecuda.bind_host_to_device(local_rank) if os.environ.get("BENCH_NO_BIND") != "1" else {"skipped": True}
    except Exception as exc:  # noqa: BLE001
        numa = {"error": repr(exc)}
    sampler = ClockSampler(local_rank) if (rank == 0 and os.environ.get("BENCH_NO_SAMPLER") != "1") else None
    if sampler:
        sampler.start()
    w0 = time.perf_counter()
    peak, peak_src = hbm_peak()
    metric, unit = METRICS[kind]
    if kind == "pir":
        import bench_pir

        threads = 8  # one step = one query on each of the `threads` concurrent host threads
        r = bench_pir.run(1 << 20, 64, threads, args.steps, cpu=not args.no_cpu_baseline)
        if r is None:
            return
        value, steps = r["value"], args.steps
        ms = r["concurrent_s"] * 1e3
        scan = r["db_scan_gbs_at_value"] / world
        roofline = {"bound": "hbm", "kernel": "inner_product_plain_kernel (first-dimension scan of the resident database)",
                    "achieved": scan, "peak": peak, "unit": "GB/s", "frac": scan / peak, "traffic": None, "peak_source": peak_src,
                    "note": "database bytes x queries/s per GPU: the scan re-reads the database once per query"}
        e2e = {"value": value, "unit": unit, "h2d_bytes_per_step": r["wire"]["unpacked_request_bytes"],
               "d2h_bytes_per_step": r["wire"]["unpacked_reply_bytes"],
               "note": "value is already end to end: every query crosses the host-pointer C ABI (query ciphertexts H2D, reply D2H)"}
    else:
        import bench_pnns

        reps = args.steps  # one step = one batch of 16 query vectors
        r = bench_pnns.run(100000, 512, 16, reps, cpu=not args.no_cpu_baseline)
        if r is None:
            return
        value, steps, ms = r["dot_products_per_s"], reps, r["batch_ms"] * reps
        scan = r["db_scan_gbs_at_value"]
        roofline = {"bound": "hbm", "kernel": "inner_product_plain_kernel (baby-step x giant-step scan of the resident matrix)",
                    "achieved": scan, "peak": peak, "unit": "GB/s", "frac": scan / peak, "traffic": None, "peak_source": peak_src,
                    "note": "matrix bytes x query vectors/s per GPU"}
        e2e = {"value": value, "unit": unit, "h2d_bytes_per_step": r["h2d_bytes_per_batch"],
               "d2h_bytes_per_step": r["d2h_bytes_per_batch"],
               "note": "value is already end to end: the query vectors cross the host-pointer C ABI every batch"}
    clocks = sampler.stop(w0, time.perf_counter()) if sampler else None
    line = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "config": {**r["config"], "workload": f"{name}: " + r["config"]["workload"], "host_numa": numa},
            "clocks": clocks, "gpu_launches": int(r["gpu_launches"]), "roofline": roofline, "cpu_baseline": r.get("cpu_baseline"),
            "e2e": e2e, "extra": {k: v for k, v in r.items() if k not in ("config", "cpu_baseline", "value", "unit", "metric")}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded sample of the last step's result to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    kind = WORKLOADS[args.workload][0]
    if args.dump_outputs and (args.impl == "reference" or kind in ("pir", "pnns")):
        ap.error("--dump-outputs covers the GPU arm of the device-resident workloads (all but C4 and C5)")

    if args.impl == "reference":
        return run_reference(args)
    if kind in ("pir", "pnns"):
        return run_app(args, args.workload)

    h = Harness(args)
    r = {"ntt": run_ntt, "mul": run_mul, "mul32": run_mul, "relin": run_relin}[kind](h, args.workload)
    if h.rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            os.sched_setaffinity(0, h.affinity0)  # the CPU arm gets every host thread, not only the GPU's NUMA node
            v, cores, sample, dt = cpu_reference_throughput(kind, r["n"], r["moduli"], r["t"])
            cpu = {"value": v, "unit": METRICS[kind][1], "cores": cores, "kind": "port", "cpu_quota_cores": cpu_quota(),
                   "sample": f"{sample} units of the same workload in {dt:.1f} s, OpenMP over units "
                             "(C restatement of the Swift reference; no Swift toolchain on this box)"}
        metric, unit = METRICS[kind]
        if kind == "ntt":
            metric = f"forward NTT/s (PolyRq.forwardNtt) at N={r['n']}, one 55-bit modulus"
        line = {
            "metric": metric, "value": r["value"], "unit": unit, "n_gpus": h.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms"] / args.steps, "higher_is_better": True, "scaling": r["scaling"], "vs_baseline": None,
            "dtype": "u32" if kind == "mul32" else "u64", "data": "synthetic", "config": r["config"], "clocks": r["clocks"],
            "gpu_launches": r["launches"],
            "roofline": r["roofline"], "cpu_baseline": cpu, "e2e": r["e2e"], "extra": r["extra"],
        }
        print(json.dumps(line))
    h.finish()


if __name__ == "__main__":
    main()
