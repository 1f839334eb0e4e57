#!/usr/bin/env python
"""bench.py -- headline metric of BASELINE.json: SGEMM TFLOP/s (2*M*N*K / t) at M=N=K=8192.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  (N > 1: launched by torch.distributed.run, one rank per GPU)

--dump-outputs DIR writes the C of the last timed step (the array the caller of the headline path receives) as
DIR/C.npy (DIR/C_rank<r>.npy per rank at N > 1), float32: the same seeded sample of DUMP_ROWS rows in every run, 32 MB
in all.  The inputs are seeded, so two builds given the same arguments can be compared output for output.

A "step" is one pass of the hot path: C <- A x B, fp32, row-major, alpha=1, beta=0 (the call the reference's bench
makes, benchmarks/gemm/gemm_bench_float32.nim:184-189), through the C ABI of liblaser_b200.so in its DEFAULT fp32 mode
(F16X3: tcgen05 kind::f16 over two fp16 pieces of the scaled operands, three passes, parity-gated at 1e-4).  At N GPUs
the headline line is weak-scaling: every rank owns 8192 rows of A and C, and each step includes B travelling over NCCL from
rank 0 (prepared there, sent in column panels), issued by the library itself (laser_b200_gemm_rowsharded_f32_dev).

One JSON line on stdout (rank 0).  Extra keys beyond the driver's contract:
  roofline       dominant kernel (gemm_tc_kernel, F16X3) against the tensor roofline
  parity         every rank checks sampled rows of ITS C panel of the timed configuration against the CPU restatement of
                 the reference (so a scaling record carries correctness, not only speed); a failed check exits non-zero
  strong_m32768  BASELINE.json config 5 in the same run: FIXED global M = 32768 (N = K = 8192) split over the ranks --
                 at --gpus 1 it is the single-GPU time of that problem, so value(N) / value(1) is the measured speed-up
  cpu_baseline   the reference CPU path (C restatement, oracle/) timed on this box's cores
  modes          (N = 1) device-resident TFLOP/s of the other kernel families and of BASELINE.json's configs 2 and 3
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "sgemm_tflops_m8192_n8192_k8192"
UNIT = "TFLOP/s"
MNK = 8192
STRONG_M = 32768
DUMP_ROWS = 1024      # rows of C written by --dump-outputs, over all ranks: 1024 x 8192 fp32 = 32 MB


def dump_rows(M, world):
    """indices of the rows of one rank's C that --dump-outputs writes: the same seeded sample in every run"""
    import numpy as np
    return np.sort(np.random.default_rng(0).choice(M, DUMP_ROWS // world, replace=False))


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the default kernel at 8192^3, from the committed
    single-pass ncu capture (profiles/r02_traffic.json names the capture file it was read from); None if absent."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(path):
        return None, None
    t = json.load(open(path))
    return float(t["dram_bytes_read"]) + float(t["dram_bytes_write"]), t.get("source")


def load_peaks():
    """MEASURED_PEAKS.json (driver-written).  The fp32 path runs on the tensor pipe whose TF32 rate is half the bf16 /
    fp16 rate (UMMA K = 8 vs 16 per instruction at the same issue rate), so the fp32 tensor-core peak is taken as
    measured bf16 / 2."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(bf16=float(p["bf16_tflops"]), bf16_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                    hbm=float(p["hbm_gbs"]), source="measured")
    return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback")  # B200_PROFILING.md


class ClockSampler:
    """nvidia-smi samples during the timed region (recipe of B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # under-load samples: the upper half of the power readings
        order = sorted(range(len(sm)), key=lambda i: pw[i])
        load = [sm[i] for i in order[len(order) // 2:]] or sm
        load.sort()
        return {"sm_mhz": load[len(load) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------- reference arm
def host_cpu_budget():
    """What this process may actually use of the host: logical CPUs, the scheduler affinity mask, and the cgroup CPU quota
    (cgroup v2 cpu.max "quota period", v1 cfs_quota_us / cfs_period_us).  A GPU lease with a CPU quota runs the same 64
    threads several times slower than an unconstrained box -- the baseline must say which it saw."""
    info = {"logical_cpus": os.cpu_count() or 1}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = info["logical_cpus"]
    quota = None
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        info["cgroup_cpu_max"] = "%s %s" % (q, p)
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            info["cgroup_cpu_max"] = "%d %d" % (q, p)
            if q > 0:
                quota = q / float(p)
        except Exception:
            info["cgroup_cpu_max"] = "unreadable"
    info["cgroup_cpu_quota"] = quota
    usable = min(info["logical_cpus"], info["affinity"])
    if quota is not None:
        usable = max(1, min(usable, int(quota + 0.5)))
    info["usable_cpus"] = usable
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                info["cpu_model"] = ln.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return info


def cpu_reference_sample(budget_s=12.0):
    """Times the structure-faithful C restatement of the reference's CPU gemm_strided (oracle/laser_cpu_gemm.c: packing +
    14x32 AVX-512 micro-kernel + OpenMP) on a bounded sample of the workload.  The OpenMP team size is calibrated first
    (usable CPUs -- affinity and cgroup quota taken into account -- vs half of them, whichever is faster on a 2048^3 probe:
    the reference's ic/jr task structure collapses when hyper-threads oversubscribe it), then the largest n in {2048, 4096,
    8192} whose run is predicted to fit the budget is timed.  Flop accounting as the reference's bench
    (gemm_common.nim:20-25)."""
    import numpy as np
    import oracle as O
    isa = O.detect_isa()
    host = host_cpu_budget()
    usable = host["usable_cpus"]

    def run(n, reps):
        a = O.fill_uniform_f32(n * n, 42, -0.1, 0.1); b = O.fill_uniform_f32(n * n, 43, -0.1, 0.1)
        c = np.zeros(n * n, np.float32)
        O.cpu_gemm_strided_f32(n, n, n, 1.0, a, n, 1, b, n, 1, 0.0, c, n, 1)      # warm-up
        ts = []
        for _ in range(reps):
            c[:] = 0                                                              # zeroed outside the timed region
            t0 = time.perf_counter()
            O.cpu_gemm_strided_f32(n, n, n, 1.0, a, n, 1, b, n, 1, 0.0, c, n, 1)
            ts.append(time.perf_counter() - t0)
        return sum(ts) / len(ts), min(ts)

    cands = sorted({usable, max(1, usable // 2)}, reverse=True)
    best_t, threads, probe = None, cands[0], {}
    for t in cands:
        O.set_num_threads(t)
        mean, _ = run(2048, 2)
        probe[str(t)] = 2 * 2048**3 / mean / 1e12
        if best_t is None or mean < best_t:
            best_t, threads = mean, t
    O.set_num_threads(threads)
    rate = 2 * 2048**3 / best_t
    n = 2048
    for cand in (4096, 8192):
        # larger problems run at a higher rate (more ic blocks per thread): x2 is conservative
        if 2 * cand**3 / (2 * rate) * 2.5 <= budget_s:
            n = cand
    reps = 3 if n < 8192 else 2
    mean, best = run(n, reps) if n != 2048 else run(2048, 5)
    tflops = 2 * n**3 / mean / 1e12
    return dict(value=tflops, unit=UNIT, cores=threads, kind="port", sample_n=n,
                sample="SGEMM %d^3 fp32 row-major (a bounded sample of the 8192^3 workload), mean of %d run(s) after 1 warm-up, "
                       "%d OpenMP threads, %s micro-kernel; C restatement of the reference (Nim is not installable here)"
                       % (n, reps, threads, O.ISA_NAMES[isa]),
                host=host, team_probe_tflops_2048=probe, ms=mean * 1e3, n=n)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    import oracle as O
    base = cpu_reference_sample(budget_s=float(os.environ.get("LASER_B200_REF_BUDGET_S", "20")))
    n = base["n"]
    a = O.fill_uniform_f32(n * n, 42, -0.1, 0.1); b = O.fill_uniform_f32(n * n, 43, -0.1, 0.1)
    c = np.zeros(n * n, np.float32)
    for _ in range(min(args.warmup, 2)):
        O.cpu_gemm_strided_f32(n, n, n, 1.0, a, n, 1, b, n, 1, 0.0, c, n, 1)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.cpu_gemm_strided_f32(n, n, n, 1.0, a, n, 1, b, n, 1, 0.0, c, n, 1)
    dt = (time.perf_counter() - t0) / args.steps
    v = 2 * n**3 / dt / 1e12
    if not (v == v and v > 0 and v != float("inf")):
        raise SystemExit("reference arm: non-finite throughput %r" % v)
    cb = dict(base); cb.pop("ms"); cb.pop("n"); cb["value"] = v
    emit({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic U(-0.1,0.1), counter-based, seed 42",
        "sample_n": n,
        "config": {"workload": "SGEMM fp32 C=A*B, per-GPU M=8192 N=K=8192 row-major, alpha=1 beta=0",
                   "timed_sample": "each step = one %d^3 product on the host CPU (TFLOP/s is size-independent accounting: 2*n^3 / t)" % n,
                   "impl": "C restatement of laser gemm_strided (oracle/), OpenMP, %d threads" % cb["cores"]},
        "cpu_baseline": cb,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


# ------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import laser_b200 as L
    import oracle as O
    from laser_b200 import rowshard as RS

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L.init()
    assert L.get_f32_mode() == L.PATH_F16X3, "bench.py measures the default fp32 mode: unset LASER_B200_F32_MODE"
    comm = RS.comm_from_torch_distributed() if world > 1 else None     # NCCL communicator owned by the library
    peaks = load_peaks()
    N = K = MNK
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / steps

    def make_problem(M_local, seed_a):
        """device-resident A (this rank's rows), B (valid on rank 0 only: NaN elsewhere until the broadcast) and C"""
        A = torch.empty(M_local * K, dtype=torch.float32, device=dev); B = torch.empty(K * N, dtype=torch.float32, device=dev)
        C = torch.empty(M_local * N, dtype=torch.float32, device=dev)
        L.fill_uniform_f32(A, M_local * K, seed_a, -0.1, 0.1)
        if rank == 0:
            L.fill_uniform_f32(B, K * N, 43, -0.1, 0.1)
        else:
            B.fill_(float("nan"))
        return A, B, C

    def make_step(M_local, A, B, C):
        A2, B2, C2 = A.view(M_local, K), B.view(K, N), C.view(M_local, N)
        if world == 1:
            return lambda: L.gemm_strided(M_local, N, K, 1.0, A, K, 1, B, N, 1, 0.0, C, N, 1)
        return lambda: RS.gemm_rowsharded(M_local, N, K, 1.0, A2, B2, 0.0, C2, src=0, comm=comm)

    def parity_check(M_local, A, B, C, rows_per_rank=16):
        """sampled rows of this rank's C panel against the CPU restatement of the reference (bit-equal to the numerics
        oracle, tests/test_oracle.py); errors are the max over ranks.  S inputs: normwise and the reference's own
        mean_relative_error (error_functions.nim:6-26) carry the gate; max-elementwise is reported for information."""
        torch.cuda.synchronize()
        rows = np.unique(np.random.default_rng(1234 + rank).integers(0, M_local, rows_per_rank))
        idx = torch.as_tensor(rows, device=dev)
        a = np.ascontiguousarray(A.view(M_local, K)[idx].cpu().numpy())
        # B is an input that lives on rank 0 (the library sends it prepared, in panels): the checker fetches the root's copy
        Bchk = B.clone()
        if world > 1:
            dist.broadcast(Bchk, src=0)
        b = Bchk.view(K, N).cpu().numpy()
        del Bchk
        got = C.view(M_local, N)[idx].cpu().numpy()
        want = np.zeros((len(rows), N), np.float32)
        O.cpu_gemm_strided_f32(len(rows), N, K, 1.0, a.reshape(-1), K, 1, b.reshape(-1), N, 1, 0.0, want.reshape(-1), N, 1)
        finite = bool(np.isfinite(got).all() and np.isfinite(b).all())
        nw = float(O.normwise_relative_error(got, want)) if finite else 1e30
        mre = float(O.mean_relative_error(got, want)) if finite else 1e30
        t = torch.tensor([nw, mre, 0.0 if finite else 1.0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        nw, mre, bad = t.tolist()
        ok = bad == 0.0 and nw < 2e-6 and mre <= 1e-5
        if bad != 0.0:
            nw = mre = None      # non-finite output (or B never arrived): strict JSON has no Infinity
        return {"rows_per_rank": int(len(rows)), "ranks": world, "normwise": nw, "mean_relative_error": mre, "ok": bool(ok),
                "gates": "normwise < 2e-6, mean_relative_error <= 1e-5 (gemm_bench_float32.nim:365-367) on every rank's rows",
                "against": "oracle/laser_cpu_gemm.c (CPU restatement of the reference, bit-equal to the numerics oracle)"}

    # ---- the metric: device-resident, default (fp32-faithful) mode, 8192 rows per rank ------------
    M = MNK
    A, B, C = make_problem(M, 42 + rank)
    step = make_step(M, A, B, C)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()       # before the warm-up so that nvidia-smi is already streaming
    for _ in range(args.warmup):
        step()
    barrier()
    n0 = L.launch_count()
    ms_step = timed(step, args.steps, 0)
    launches = L.launch_count() - n0
    dump = None
    if args.dump_outputs:
        # read before the profiled and untimed steps below run the product again
        dump = C.view(M, N)[torch.as_tensor(dump_rows(M, world), device=dev)].cpu().numpy()
    # kernel-level roofline numbers: the same step, bracketed by CUDA events inside the library (profile mode disables the
    # dependent launch of the GEMM kernel, so it is measured separately from the headline time above)
    L.profile_begin()
    prof_steps = max(3, min(args.steps, 10))
    for _ in range(prof_steps):
        step()
    prof = L.profile_end()
    # nvidia-smi samples every 100 ms; if the timed region was shorter than ~1.5 s keep the very same step running
    # (untimed) so that the clock/throttle record is under this load
    obs_steps = int(max(0.0, 1500.0 - ms_step * (args.steps + prof_steps)) / max(ms_step, 1e-3))
    if world > 1:
        t_obs = torch.tensor([obs_steps], device=dev)
        dist.broadcast(t_obs, src=0)
        obs_steps = int(t_obs.item())
    for _ in range(obs_steps):
        step()
    barrier()
    clocks = sampler.stop() if sampler else None
    if clocks is not None:
        clocks["observed_over"] = "warm-up + %d timed + %d profiled + %d untimed identical steps" % (args.steps, prof_steps, obs_steps)
    parity = parity_check(M, A, B, C)
    flops_step = 2.0 * M * N * K * world
    value = flops_step / (ms_step * 1e-3) / 1e12

    roofline = None
    if rank == 0:
        gemm_ms = prof["gemm_ms"] / max(1, prof["gemm_launches"])
        flops_launch = 2.0 * M * N * K / max(1, prof["gemm_launches"] // prof_steps)   # algorithmic flops of one launch
        achieved = flops_launch / (gemm_ms * 1e-3) / 1e12
        tf32_peak = peaks["bf16"] / 2.0
        traffic, traffic_src = load_traffic()
        roofline = {"bound": "tensor", "kernel": "gemm_tc_kernel<fp16 pieces, 3 passes, CTA pair, scaled epilogue> (F16X3)",
                    "achieved": achieved, "peak": tf32_peak, "unit": "TFLOP/s", "frac": achieved / tf32_peak,
                    "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst) / 2 = fp32 (TF32-rate) tensor peak, of %s" % peaks["source"],
                    "tensor_pipe_frac": 1.5 * achieved / tf32_peak,
                    "frac_of_sustained_peak": achieved / (peaks["bf16_sustained"] / 2.0),
                    "sustained_note": "kernel_ms is the CUDA-event time of the kernel inside a long back-to-back sequence (the part is at its power "
                                      "cap by then); B200_PROFILING.md pairs such a time with the SUSTAINED cuBLAS figure (bf16_tflops_sustained / 2): "
                                      "frac_of_sustained_peak.  `frac` keeps the stricter burst denominator used in round 1",
                    "note": "achieved counts ALGORITHMIC flops 2MNK; the default mode issues three fp16 MMAs (K = 16 each, the bf16 "
                            "rate) per useful MAC = 1.5 TF32-equivalents, so frac <= 2/3 by construction and tensor_pipe_frac = "
                            "1.5 * frac is the tensor-pipe utilisation; traffic = ncu dram bytes read + written per launch "
                            "(committed single-pass capture), algorithmic bytes = 805 MB",
                    "kernel_ms": gemm_ms, "prep_ms_per_step": prof["prep_ms"] / prof_steps,
                    "step_frac": (2.0 * M * N * K / (ms_step * 1e-3) / 1e12) / tf32_peak if world == 1 else None}

    # ---- BASELINE.json config 5 in the same run: fixed global M = 32768 over the ranks (strong scaling) ----
    del A, C
    lo, hi = RS.partition_rows(STRONG_M, world)[rank]
    Ms = hi - lo
    As = torch.empty(max(Ms, 1) * K, dtype=torch.float32, device=dev); Cs = torch.empty(max(Ms, 1) * N, dtype=torch.float32, device=dev)
    L.fill_uniform_f32(As, max(Ms, 1) * K, 142 + rank, -0.1, 0.1)
    if rank == 0:
        L.fill_uniform_f32(B, K * N, 43, -0.1, 0.1)
    else:
        B.fill_(float("nan"))
    sstep = make_step(Ms, As, B, Cs)
    s_steps = max(3, args.steps // 2)
    ms_strong = timed(sstep, s_steps, 2)
    strong_parity = parity_check(Ms, As, B, Cs, rows_per_rank=8) if Ms > 0 else None
    strong = {"global_M": STRONG_M, "N": N, "K": K, "rows_per_rank": Ms, "ms_per_step": ms_strong, "steps": s_steps,
              "value": 2.0 * STRONG_M * N * K / (ms_strong * 1e-3) / 1e12, "unit": UNIT, "scaling": "strong",
              "parity": strong_parity,
              "note": "same call as the headline (row-sharded, B travels over NCCL from rank 0 every step at N > 1); speed-up at N GPUs = "
                      "this value at --gpus N / this value at --gpus 1"}
    del As, Cs

    # ---- informational: the other kernel families and BASELINE.json's configs 2 / 3, device-resident ----
    modes = {}
    if world == 1:
        A = torch.empty(M * K, dtype=torch.float32, device=dev); C = torch.empty(M * N, dtype=torch.float32, device=dev)
        L.fill_uniform_f32(A, M * K, 42, -0.1, 0.1)
        half = max(3, args.steps // 2)
        ms1 = timed(lambda: L.gemm_strided(M, N, K, 1.0, A, K, 1, B, N, 1, 0.0, C, N, 1, path=L.PATH_TF32X1), half, 2)
        ms3 = timed(lambda: L.gemm_strided(M, N, K, 1.0, A, K, 1, B, N, 1, 0.0, C, N, 1, path=L.PATH_TF32X3), half, 2)
        modes["tf32x3_any_range"] = {"tflops": 2.0 * M * N * K / ms3 / 1e9, "ms": ms3,
                                     "note": "three tf32 passes over hi/lo pieces: fp32-faithful without the row/column scaling of the default mode"}
        modes["tf32x1_fast_mode"] = {"tflops": 2.0 * M * N * K / ms1 / 1e9, "ms": ms1, "tolerance": "normwise 2e-3 (hardware truncates fp32 -> tf32)",
                                     "frac_of_tf32_peak": 2.0 * M * N * K / ms1 / 1e9 / (peaks["bf16"] / 2.0),
                                     "note": "TMA reads the caller's fp32 memory directly: no preparation pass at all"}
        Ab = A.view(M, K).to(torch.bfloat16); Bb = B.view(K, N).to(torch.bfloat16); Cb = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
        msb = timed(lambda: L.gemm_strided(M, N, K, 1.0, Ab, K, 1, Bb, N, 1, 0.0, Cb, N, 1), half, 2)
        modes["bf16_8192_config4"] = {"tflops": 2.0 * M * N * K / msb / 1e9, "ms": msb, "frac_of_bf16_peak": 2.0 * M * N * K / msb / 1e9 / peaks["bf16"]}
        del Ab, Bb, Cb
        n4 = 4096
        a4, b4, c4 = A[:n4 * n4], B[:n4 * n4], C[:n4 * n4]
        ms4 = timed(lambda: L.gemm_strided(n4, n4, n4, 1.0, a4, n4, 1, b4, n4, 1, 0.0, c4, n4, 1), 2 * half, 3)
        ms4t = timed(lambda: L.gemm_strided(n4, n4, n4, 1.0, a4, 1, n4, b4, n4, 1, 0.0, c4, n4, 1), 2 * half, 3)
        modes["f32_4096_config2"] = {"tflops": 2.0 * n4**3 / ms4 / 1e9, "ms": ms4, "layout": "A, B row-major"}
        modes["f32_4096_At_config3"] = {"tflops": 2.0 * n4**3 / ms4t / 1e9, "ms": ms4t,
                                        "layout": "A given transposed (rowStrideA = 1, colStrideA = M): MN-major TMA tiles, no physical transpose"}
        # fp64 of the same entry point (gemm.nim:234-246): FP64 tensor cores (mma.sync DMMA), bit-identical to the reference's FMA chain
        n64 = 4096
        a64 = torch.rand(n64, n64, dtype=torch.float64, device=dev) - 0.5; b64 = torch.rand(n64, n64, dtype=torch.float64, device=dev) - 0.5
        c64 = torch.empty(n64, n64, dtype=torch.float64, device=dev)
        ms64 = timed(lambda: L.gemm_strided(n64, n64, n64, 1.0, a64, n64, 1, b64, n64, 1, 0.0, c64, n64, 1), 3, 1)
        modes["f64_4096_dmma"] = {"tflops": 2.0 * n64**3 / ms64 / 1e9, "ms": ms64, "note": "float64 gemm_strided on the FP64 tensor cores, bit-exact vs the oracle"}
        del a64, b64, c64
        del A, C

    # ---- e2e: the drop-in call with HOST buffers, copies inside the timed region ----------------
    hA = torch.empty(M * K, dtype=torch.float32).pin_memory(); hB = torch.empty(K * N, dtype=torch.float32).pin_memory()
    hC = torch.empty(M * N, dtype=torch.float32).pin_memory()
    gA = torch.empty(M * K, dtype=torch.float32, device=dev)
    L.fill_uniform_f32(gA, M * K, 42 + rank, -0.1, 0.1)
    hA.copy_(gA.cpu()); del gA
    if world > 1:
        dist.broadcast(B, src=0)   # every rank's own host-pointer call needs a valid B (the row-sharded steps above do not deliver it)
    hB.copy_(B.cpu())
    nA, nB, nC = hA.numpy(), hB.numpy(), hC.numpy()
    e2e_steps = max(2, min(args.steps, 5))
    L.gemm_strided(M, N, K, 1.0, nA, K, 1, nB, N, 1, 0.0, nC, N, 1)     # warm-up (staging buffers)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        L.gemm_strided(M, N, K, 1.0, nA, K, 1, nB, N, 1, 0.0, nC, N, 1)  # synchronous: C valid on the host at return
    t1 = time.perf_counter()
    e2e_ms = torch.tensor([(t1 - t0) * 1e3 / e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e = {"value": flops_step / (e2e_ms.item() * 1e-3) / 1e12, "unit": UNIT, "ms_per_step": e2e_ms.item(),
           "h2d_bytes_per_step": (M * K + K * N) * 4 * world, "d2h_bytes_per_step": M * N * 4 * world,
           "api": "laser_b200_gemm_strided_f32 (host pointers, reference signature), pinned host buffers, steps=%d" % e2e_steps}

    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "C.npy" if world == 1 else "C_rank%d.npy" % rank), dump)

    ok = parity["ok"] and (strong_parity is None or strong_parity["ok"])
    if rank == 0:
        cpu = cpu_reference_sample() if world == 1 else None
        if cpu:
            cpu.pop("ms"); cpu.pop("n")
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic U(-0.1,0.1), counter-based generator, seed 42 (device-generated)",
            "config": {"workload": "SGEMM fp32 C=A*B, per-GPU M=8192 N=K=8192 row-major, alpha=1 beta=0"
                                   + ("" if world == 1 else "; row-sharded: total M=%d, B travels over NCCL from rank 0 every step (prepared fp16 pieces + scales, column panels) "
                                                            "(laser_b200_gemm_rowsharded_f32_dev)" % (M * world)),
                       "global_M": M * world, "N": N, "K": K, "parallelism": "rowshard%d" % world,
                       "f32_mode": "f16x3 (fp32-faithful, default)", "l2": "inputs larger than L2 (A+B+C = 805 MB vs 126 MB)",
                       "timing": "CUDA events on the launching stream, barrier + synchronize both sides, max over ranks"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "parity": parity,
            "strong_m32768": strong,
        }
        if cpu:
            out["cpu_baseline"] = cpu
        out["modes"] = _finite_json(modes)     # informational legs only: a non-finite number there must not take the line down
        emit(out)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not ok:
        raise SystemExit("bench.py: PARITY FAILED (see the 'parity' / 'strong_m32768.parity' keys of the line)")


def _finite_json(x):
    """non-finite numbers -> None, recursively (applied to the informational `modes` sub-dict only)"""
    import math
    if isinstance(x, float):
        return x if math.isfinite(x) else None
    if isinstance(x, dict):
        return {k: _finite_json(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_finite_json(v) for v in x]
    return x


class StdoutGuard:
    """Only the result line may reach stdout: native libraries (NCCL prints its version banner
    to stdout) get fd 1 redirected to stderr for the duration of the run."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line):
        sys.stdout.flush()
        os.write(self.real, (line + "\n").encode())


GUARD = None


def emit(obj):
    # strict JSON: a non-finite headline number is an error, not a null (json.dumps raises ValueError)
    line = json.dumps(obj, allow_nan=False)
    if GUARD is not None:
        GUARD.emit(line)
    else:
        print(line, flush=True)


def main():
    if os.environ.get("LASER_B200_LIB") or os.environ.get("LASER_B200_EMU"):
        raise SystemExit("bench.py measures the in-tree CUDA library only: unset LASER_B200_LIB / LASER_B200_EMU")
    global GUARD
    GUARD = StdoutGuard()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the C of the last timed step (a seeded sample of rows) as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
