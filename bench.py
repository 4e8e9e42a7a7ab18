#!/usr/bin/env python
"""bench.py — bases evaluated per second by the extreme-point enumeration path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--m 12 --n 40 --seed 1]
                    [--algo auto|independent|shared] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one complete enumeration of all C(n, m) bases of one synthetic dense
LP (default: BASELINE.json's roofline headline, m=12, n=40 -> 5 586 853 480
bases).  With N > 1 (launched by torchrun, one process per GPU) rank r takes the
interleaved cost-weighted windows r, r+N, ... of the rank space — strong
scaling: the job is the same LP — and every step ends with one NCCL all_gather
of the 256-byte partial records.

Printed JSON line (rank 0):
  value     bases/s, inputs resident in HBM; K steps inside a barrier +
            cuda synchronize bracket, each timed with CUDA events on the
            launching stream (launch + all-gather), max over ranks per step;
            best and median per step are reported next to the mean
  e2e       same metric through the public host-buffer call
            (EnumerationSolver -> enumgpu_solve: H2D of A,b,c + kernels + D2H)
  roofline  FP64-pipe roofline of the enumeration kernel: algorithmic flops
            F(m) = 2/3 m^3 + 3/2 m^2 + 5/6 m per basis (SURVEY §8d) x bases per
            launch / CUDA-event time of the launch; peak = max(in-run DFMA
            probe, nominal 148 SM x 64 lanes x 2 x f_max) (MEASURED_PEAKS.json
            carries no FP64 figure)
  cpu_baseline  the CPU oracle on this box's host cores on a bounded sample

--dump-outputs DIR writes the last timed step's result records (status, best_rank, basis,
x_B, objective, counts: one row per record) as float64 DIR/<name>.npy: the merged record
of all ranks for the GPU arm, one record per sampled window for --impl reference.

--impl reference times the CPU arm only (the reference's EnumerationSolver is
an unimplemented stub and its building blocks need Eigen, which is not on the
box: the arm is oracle/enumcpu.c, kind "port").
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from simplexmethod_b200 import _abi, lpgen  # noqa: E402


def algo_flops_per_basis(m: int) -> float:
    return 2.0 / 3.0 * m ** 3 + 1.5 * m ** 2 + 5.0 / 6.0 * m


def binom(n, k):
    from math import comb
    return comb(n, k)


# ------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([v.strip() for v in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------ CPU baseline
def cpu_sample_windows(total: int, budget_ranks: int):
    """A prefix plus 8 pseudo-random windows, about budget_ranks ranks in all."""
    if total <= budget_ranks:
        return [(0, total)]
    w = budget_ranks // 12
    rng = np.random.default_rng(2026)
    wins = [(0, 4 * w)]
    for s in sorted(int(v) for v in rng.integers(4 * w, total - w, 8)):
        wins.append((s, s + w))
    return wins


def cpu_baseline(A, b, c, mx, m, n, budget_ranks, threads):
    from oracle import enumcpu
    total = binom(n, m)
    wins = cpu_sample_windows(total, budget_ranks)
    ranks, secs, results = 0, 0.0, []
    for (a, e) in wins:
        t = time.perf_counter()
        results.append(enumcpu.solve(A, b, c, mx, n_threads=threads, rank_begin=a, rank_end=e)[0])
        secs += time.perf_counter() - t
        ranks += e - a
    desc = (f"full range of {total} ranks" if len(wins) == 1 else
            f"{ranks} of {total} ranks: prefix [0,{wins[0][1]}) + 8 windows of {wins[1][1] - wins[1][0]} ranks")
    return ranks / secs, desc, ranks, secs, results


def dump_outputs(out_dir, results, m):
    """The result records of a step, one row per record, as float64 .npy files (ranks and counts are below 2^53,
    so exact).  The workload is seeded: the same arguments give the same inputs, so two builds compare file by file."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {
        "status": [r.status for r in results],
        "best_rank": [r.best_rank for r in results],
        "basis": [list(r.basis)[:m] for r in results],
        "x_B": [list(r.x_B)[:m] for r in results],
        "objective": [r.objective for r in results],
        "counts": [[r.n_bases, r.n_singular, r.n_infeasible, r.n_feasible] for r in results],
    }
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, dtype=np.float64))


def reference_code_rate(A, b, c, mx, m, n, threads, seconds=4.0):
    """Side figure for the reference arm: the enumeration composed from the reference's OWN per-basis code
    (oracle/_ref: Canonical::GetBasicSolution / IsFeasibleBasis / Evaluate + FullPivLU::isInvertible, compiled from
    /root/reference against oracle/eigen_shim) on all host threads, for a few seconds.  NOT the arm's value: the
    linear algebra under it is the shim's unoptimised code, not Eigen's, so it understates the reference."""
    try:
        from concurrent.futures import ThreadPoolExecutor
        from oracle import simplexref
        if not simplexref.available():
            return None
        total = binom(n, m)
        rng = np.random.default_rng(11)
        per = 400                                       # ranks per call (~50 ms at m=12)
        t_end = time.perf_counter() + seconds

        def work(seed):
            done, r = 0, np.random.default_rng(seed)
            while time.perf_counter() < t_end:
                lo = int(r.integers(0, max(1, total - per)))
                simplexref.enumerate_bases(A, b, c, mx, rank_begin=lo, rank_end=min(total, lo + per))
                done += min(total, lo + per) - lo
            return done

        t0 = time.perf_counter()
        with ThreadPoolExecutor(threads) as ex:
            ranks = sum(ex.map(work, [int(v) for v in rng.integers(0, 1 << 30, threads)]))
        secs = time.perf_counter() - t0
        la = simplexref.linear_algebra()
        return {"value": ranks / secs, "unit": "bases/s", "cores": threads, "sample": f"{ranks} ranks in random windows of {per}",
                "linear_algebra": la,
                "what": ("reference's own per-basis code (oracle/_ref) compiled against real Eigen: the per-basis Eigen column of BASELINE.md"
                         if la.startswith("eigen") else
                         "reference's own per-basis code (oracle/_ref) with an Eigen API stand-in for the absent Eigen: "
                         "a side figure, slower than real Eigen would be; the arm's value is the faster oracle port")}
    except Exception as e:                              # never let the side figure break the arm
        return {"unavailable": str(e)}


# ------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    # (--lp-m / --lp-n: the same options under names torchrun's own parser does not mistake for its --max-restarts ...)
    ap.add_argument("--m", "--lp-m", dest="m", type=int, default=12)
    ap.add_argument("--n", "--lp-n", dest="n", type=int, default=40)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--algo", default="auto", choices=["auto", "independent", "shared"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-ranks", type=int, default=120_000_000, help="ranks in the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the result records of the last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    m, n = args.m, args.n
    total = binom(n, m)
    A, b, c, mx = lpgen.dense_lp(m, n, args.seed)
    workload = f"dense canonical LP m={m} n={n} seed={args.seed}: full enumeration of C({n},{m})={total} bases"
    config = {"workload": workload, "m": m, "n": n, "seed": args.seed, "bases_per_step": total,
              "sharding": f"{world} shards of interleaved cost-weighted windows" if world > 1 else "single GPU",
              "l2": "inputs are (m*n+m+n)*8 bytes staged in shared memory; compute-bound, L2 state irrelevant"}

    if args.impl == "reference":
        if rank != 0:
            return
        threads = os.cpu_count() or 1
        budget = max(args.cpu_ranks // 4, 1_000_000)
        for _ in range(args.warmup):
            cpu_baseline(A, b, c, mx, m, n, budget // 8, threads)
        t_ranks, t_secs, desc, step_results = 0, 0.0, "", []
        for _ in range(args.steps):
            _, desc, r, s, step_results = cpu_baseline(A, b, c, mx, m, n, budget, threads)
            t_ranks += r; t_secs += s
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, step_results, m)     # one record per sampled window
        v = t_ranks / t_secs
        ref_code = reference_code_rate(A, b, c, mx, m, n, threads)
        kind, sample_note = "port", ("the reference's EnumerationSolver is a stub and Eigen is absent, so the arm is the "
                                     "Eigen-free oracle port (oracle/enumcpu.c)")
        if ref_code and str(ref_code.get("linear_algebra", "")).startswith("eigen") and ref_code.get("value"):
            # a box with real Eigen: the enumeration composed from the reference's own primitives IS the reference arm
            v, kind = ref_code["value"], "reference"
            sample_note = "enumeration composed from the reference's own per-basis code compiled against real Eigen (oracle/_ref); " + ref_code["sample"]
        print(json.dumps({
            "impl": "reference", "metric": "bases evaluated per second", "value": v, "unit": "bases/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_secs / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": v, "unit": "bases/s", "cores": threads, "kind": kind,
                             "sample": f"each step: {desc}; {sample_note}"},
            "e2e": {"value": v, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "reference_code": ref_code,
        }))
        return

    import torch
    import torch.distributed as dist
    import simplexmethod_b200 as sm

    L = sm.lib()
    if not torch.cuda.is_available() or L.enumgpu_device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: libenumgpu has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries the one JSON line only.  At NCCL_DEBUG=VERSION (this pool's default) NCCL prints its
        # "NCCL version ..." banner on stdout and ignores NCCL_DEBUG_FILE (honoured from WARN up): raise VERSION to
        # WARN and send NCCL's debug output to stderr
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    algo = {"auto": _abi.ALGO_AUTO, "independent": _abi.ALGO_INDEPENDENT, "shared": _abi.ALGO_SHARED}[args.algo]

    # this rank's shard (strong scaling: same LP): the interleaved windows rank, rank+world, ... of the
    # whole space (enumgpu_options.shard_index/count)
    from simplexmethod_b200 import dist as edist

    # inputs resident in HBM
    dA = torch.from_numpy(np.ascontiguousarray(A.T)).to(dev)
    db, dc = torch.from_numpy(b).to(dev), torch.from_numpy(c).to(dev)
    scale = float(np.abs(A).max())
    pd = _abi.Problem(m, n, m, int(mx), dA.data_ptr(), db.data_ptr(), dc.data_ptr())
    part = torch.zeros(256, dtype=torch.uint8, device=dev)
    gathered = torch.zeros(world * 256, dtype=torch.uint8, device=dev)
    flush = torch.empty(160 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB of L2
    nl = C.c_int32()
    handle = C.c_void_p()
    if L.enumgpu_create(local_rank, C.byref(handle)) != 0:
        raise RuntimeError(sm.last_error())
    # everything of a step — flush, events, the enumeration launch, the all-gather — goes to ONE stream, torch's
    # current one, handed to the library per call (torch.cuda.Event only sees the stream it is recorded on)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    torch.cuda.set_stream(stream)
    opt = _abi.Options(-1.0, -1.0, 0, total, 0, algo, None, stream.cuda_stream, rank if world > 1 else 0, world if world > 1 else 0)

    def enqueue_step():
        rc = L.enumgpu_enqueue_h(handle, C.byref(pd), scale, C.byref(opt), part.data_ptr(), C.byref(nl))
        if rc != 0:
            raise RuntimeError(sm.last_error())
        edist.all_gather_records(part, gathered, world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput -------------------------------------
    # A step = [L2 flush, untimed] + [enumeration launch + all-gather of the records, timed with CUDA events on the
    # launching stream].  The flush sits between the timed brackets: the path's working set is 4 KB of inputs held
    # in shared memory, so the flush changes nothing measurable, but the rule asks for it and it must not be billed
    # to the enumeration (at 8 GPUs the 160 MB fill was 0.65 % of a step).
    for _ in range(args.warmup):
        flush.fill_(1)
        enqueue_step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(1)
        ev[i][0].record(stream)
        rc = L.enumgpu_enqueue_h(handle, C.byref(pd), scale, C.byref(opt), part.data_ptr(), C.byref(nl))
        if rc != 0:
            raise RuntimeError(sm.last_error())
        ev[i][1].record(stream)
        edist.all_gather_records(part, gathered, world)
        ev[i][2].record(stream)
    barrier()
    wall_incl_flush = max_over_ranks(time.perf_counter() - t0)
    launches_per_step = nl.value                     # kernels of libenumgpu per step (the L2-flush fill and the
                                                     # NCCL all-gather / 256-byte copy are torch's and not counted)
    kern_ms = [e[0].elapsed_time(e[1]) for e in ev]  # this rank's enumeration launches (CUDA events, same stream)
    step_ms = [e[0].elapsed_time(e[2]) for e in ev]  # launch + all-gather: the timed step
    # a step ends when its all-gather has delivered every rank's record: per step, the max over ranks
    if world > 1:
        t = torch.tensor(step_ms, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        step_ms = t.cpu().tolist()
    kern_ms_own = float(np.mean(kern_ms))
    kern_ms_max = max_over_ranks(kern_ms_own)
    timed_s = 1e-3 * float(np.sum(step_ms))
    # the clock sampler covers the device-timed region only: an nvidia-smi query every 200 ms takes driver locks that
    # show up as 2 ms outliers in the host-timed e2e steps below
    clocks = sampler.stop() if rank == 0 else None
    own_bases = _abi.Partial.from_buffer_copy(part.cpu().numpy().tobytes()).n_bases
    res = edist.merge_records(gathered.cpu().numpy().tobytes(), world)     # the last timed step's records, merged
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, [res], m)
    value = total * args.steps / timed_s

    # ---- end to end through the public host-buffer API ------------------
    # N = 1: EnumerationSolver(canonical).enumerate() -> enumgpu_solve_hv (pack into pinned memory, H2D of A|b|c,
    # one kernel, D2H of the 256-byte record, synchronise).  N > 1: dist.ShardedEnumeration.solve(), the same per
    # rank plus the device-side all-gather and one D2H of the gathered records.
    can = sm.Canonical(A, b, c, list(range(m)), minimize=not mx)
    if world == 1:
        solver = sm.EnumerationSolver(can, algo=algo)
        step_e2e = lambda: solver.enumerate()
        h2d, d2h = (m * n + m + n) * 8, 256
    else:
        sharded = edist.ShardedEnumeration(local_rank, rank, world, algo)
        step_e2e = lambda: sharded.solve(A, b, c, mx)
        h2d, d2h = (m * n + m + n) * 8, 256 * world
    for _ in range(max(2, args.warmup)):
        r_e2e = step_e2e()
    barrier()
    e2e_times = []
    for _ in range(args.steps):
        barrier()
        t0 = time.perf_counter()
        r_e2e = step_e2e()
        e2e_times.append(time.perf_counter() - t0)
    barrier()
    if world > 1:
        t = torch.tensor(e2e_times, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_times = t.cpu().tolist()
    e2e_s = float(np.sum(e2e_times))
    e2e_value = total * args.steps / e2e_s
    assert (r_e2e.best_rank, r_e2e.n_feasible, r_e2e.n_singular) == (res.best_rank, res.n_feasible, res.n_singular)

    if world > 1:
        dist.barrier()
    if rank != 0:
        # (the handle is left to process teardown: torch still holds tensors that were allocated on its stream)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the enumeration launch ------------------------------
    F = algo_flops_per_basis(m)
    probe_detail = (C.c_double * 2)(0.0, 0.0)
    probe = L.enumgpu_fp64_peak_detail(3, probe_detail)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    sm_max = float((clocks or {}).get("sm_max_mhz") or peaks.get("sm_max_mhz", 1965.0))
    nominal = 148 * 64 * 2 * sm_max * 1e6 / 1e12
    peak = max(probe, nominal)                  # the larger of the two: never flatter the kernel with a low probe
    shard = own_bases                           # bases this rank's launch visited
    achieved = shard * F / (kern_ms_own * 1e-3) / 1e12
    kernel_name = "k_shared" if res.algo_used == _abi.ALGO_SHARED else "k_independent"
    # the "one LU per basis" kernel on a bounded sample, for the same roofline: what the FP64 pipe does
    # when nothing is shared or pruned (ENUMGPU_ALGO_INDEPENDENT, same arithmetic, same results)
    indep = None
    if world == 1 and res.algo_used == _abi.ALGO_SHARED:
        sample = min(total, 200_000_000)
        opt_i = _abi.Options(-1.0, -1.0, 0, sample, 0, _abi.ALGO_INDEPENDENT, None, stream.cuda_stream)
        res_i = _abi.Result()
        for _ in range(2):
            if L.enumgpu_solve_device(C.byref(pd), scale, C.byref(opt_i), C.byref(res_i)) != 0:
                raise RuntimeError(sm.last_error())
        ach_i = sample * F / (res_i.kernel_ms * 1e-3) / 1e12
        indep = {"kernel": "k_independent", "sample_ranks": sample, "launch_ms": res_i.kernel_ms,
                 "bases_per_s": sample / (res_i.kernel_ms * 1e-3), "achieved": ach_i, "frac": ach_i / peak}
    # executed (not algorithmic) work and DRAM traffic of the kernel: ONLY from an ncu capture of this very kernel —
    # the key-metrics file under profiles/ is used iff its recorded launch time is within 3 % of the launch time
    # measured in this run (same code, same configuration); otherwise these fields are null, never stale constants
    executed, traffic, profile_note = None, None, None
    prof = os.path.join(ROOT, "profiles", f"r2_{kernel_name}_m{m}n{n}_ncu_key_metrics.csv")
    if world == 1 and os.path.exists(prof):
        kv, unit_of = {}, {}
        for line in open(prof):
            f = line.rstrip("\n").split(",")
            if len(f) >= 3:
                try:
                    kv[f[0]] = float(f[2])
                    unit_of[f[0]] = f[1]
                except ValueError:
                    pass
        to_ms = {"ns": 1e-6, "us": 1e-3, "ms": 1.0, "s": 1e3}
        to_bytes = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        if "gpu__time_duration.sum" in kv:
            kv["gpu__time_duration.sum"] *= to_ms.get(unit_of["gpu__time_duration.sum"], 1.0)
        t_prof = kv.get("gpu__time_duration.sum")
        if t_prof and abs(t_prof - kern_ms_own) <= 0.03 * kern_ms_own:
            fpb = kv.get("derived_executed_flops_per_basis")
            if fpb:
                ex = shard * fpb / (kern_ms_own * 1e-3) / 1e12
                executed = {"flops_per_basis": fpb, "tflops": ex, "frac_of_peak": ex / peak,
                            "warp_instructions_per_basis": kv.get("derived_warp_inst_per_basis"),
                            "fp64_pipe_busy_pct": kv.get("sm__inst_executed_pipe_fp64.avg.pct_of_peak_sustained_active"),
                            "issue_slots_busy_pct": kv.get("smsp__issue_active.avg.pct_of_peak_sustained_active"),
                            "from_profile": os.path.relpath(prof, ROOT), "profile_launch_ms": t_prof}
            rd, wr = kv.get("dram__bytes_read.sum"), kv.get("dram__bytes_write.sum")
            if rd is not None and wr is not None:
                traffic = int(round(rd * to_bytes.get(unit_of["dram__bytes_read.sum"], 1.0) +
                                    wr * to_bytes.get(unit_of["dram__bytes_write.sum"], 1.0)))
        else:
            profile_note = (f"{os.path.relpath(prof, ROOT)} records a {t_prof} ms launch, this run measured {kern_ms_own:.3f} ms: "
                            "more than 3 % apart, so executed/traffic are not quoted")
    roofline = {"bound": "fp64", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic,
                "traffic_unit": "bytes per launch, dram__bytes_read.sum + dram__bytes_write.sum of the ncu capture named in "
                                "executed.from_profile (algorithmic input: (m*n+m+n)*8 bytes; the rest is instruction fetch, "
                                "tables, spill write-back); null when no capture matches this build",
                "peak_source": "max(in-run register-resident DFMA-chain probe, nominal 148 SM x 64 lanes x 2 x f_max); "
                               "MEASURED_PEAKS.json has no FP64 figure",
                "peak_probe": probe, "peak_nominal": nominal,
                "peak_probe_detail": {"sm_mhz_during_probe": probe_detail[1],
                                      "dfma_warp_instr_per_sm_cycle": (probe * 1e12 / (2 * 32 * 148 * probe_detail[1] * 1e6)) if probe_detail[1] else None,
                                      "note": "the pipe issues at most 2 DFMA warp-instructions per SM cycle (1.98 measured on one SM alone, "
                                              "profiles/r1_fp64_micro.txt); with all 148 SMs busy the chip sustains the rate given here at the "
                                              "clock given here (clock64 against globaltimer inside the probe): the probe is below nominal "
                                              "because of the issue rate, not the clock"},
                "flops_per_basis": F, "bases_per_launch": shard, "launch_ms": kern_ms_own,
                "launch_ms_best": float(np.min(kern_ms)), "launch_ms_median": float(np.median(kern_ms)),
                "launch_ms_max_over_ranks": kern_ms_max, "kernel": kernel_name,
                "executed": executed, "profile_note": profile_note, "per_basis_lu_kernel": indep,
                "note": "achieved/frac are ALGORITHMIC flops (one dgesv + dot per basis, SURVEY 8d); k_shared shares the "
                        "first m-4 elimination steps between bases and prunes the back substitution, so frac > 1 is "
                        "expected: 'executed' is what the FP64 pipe really did, 'per_basis_lu_kernel' the kernel "
                        "that does one full LU per basis (DESIGN.md 5-6)"}

    config["l2"] = ("inputs are (m*n+m+n)*8 bytes staged in shared memory; compute-bound, L2 state irrelevant; a 160 MB "
                    "buffer (L2 is 126 MB) is rewritten between the timed steps, outside the CUDA-event brackets")
    config["timing"] = ("per step: CUDA events on the launching stream around [enumeration launch + all-gather of the 256-byte "
                        "records]; per step the max over ranks; value = bases x steps / sum of the steps")
    out = {
        "metric": "bases evaluated per second", "value": value, "unit": "bases/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * timed_s / args.steps,
        "ms_per_step_best": float(np.min(step_ms)), "ms_per_step_median": float(np.median(step_ms)),
        "wall_ms_per_step_incl_flush": 1e3 * wall_incl_flush / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config,
        "e2e": {"value": e2e_value, "unit": "bases/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * e2e_s / args.steps, "ms_per_step_best": 1e3 * float(np.min(e2e_times)),
                "ms_per_step_median": 1e3 * float(np.median(e2e_times)),
                "api": "EnumerationSolver.enumerate -> enumgpu_solve_hv" if world == 1 else
                       "dist.ShardedEnumeration.solve -> enumgpu_enqueue_h + NCCL all-gather"},
        "gpu_launches": launches_per_step * args.steps,
        "clocks": clocks, "roofline": roofline,
        "result": {"status": res.status, "best_rank": res.best_rank, "basis": list(res.basis)[:m],
                   "objective": res.objective, "n_singular": res.n_singular, "n_infeasible": res.n_infeasible,
                   "n_feasible": res.n_feasible, "algo_used": res.algo_used},
    }
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, desc, _, _, _ = cpu_baseline(A, b, c, mx, m, n, args.cpu_ranks, threads)
        out["cpu_baseline"] = {"value": v, "unit": "bases/s", "cores": threads, "kind": "port",
                               "sample": desc + "; Eigen-free oracle port (the reference path is a stub and Eigen is absent)"}
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
