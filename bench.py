#!/usr/bin/env python
"""bench.py -- throughput of the Heston path-simulation hot path on N B200s (one process per GPU).

Contract: `python bench.py --gpus N --steps K --warmup W` (N>1: launched by torch.distributed.run) prints ONE
JSON line on rank 0.  A "step" is one compute() pass of the hot path over one batch of synthetic paths.
`--steps K` sets the timed steps of the headline and of the em sub-record; the other sub-records time fixed counts (below).

Headline (the line's own metric/value): BASELINE.json configs[1] -- FE Euler, N=1000 time steps, 2^24 paths per GPU,
README parameters, seed 1234.  Paths shard over ranks by disjoint Philox subsequences (weak scaling); one NCCL
allreduce of the two FP64 moments per step when N>1.

`--dump-outputs DIR` writes what each timed path returned in its last timed step, the FP64 sums (payoff, payoff^2), as
DIR/<name>.npy: `moments` (headline), and with the sub-records `em_moments`, `c5_fe_moments`, `c5_em_moments` and
`c4_fe_moments` / `c4_em_moments` (one row per grid point).  Seeds are fixed, so the same arguments give the same inputs
and two builds can be compared output for output.

  value     FE: path-steps/s, whole job; inputs are 11 scalars (nothing to stage in HBM)
  e2e       the same metric through the public C-ABI call nmch_engine_compute() with host buffers:
            kernel-parameter upload + launch + sync + the result landing in host memory, every step
  roofline  the FE kernel against the FP32/SFU ISSUE roofline of SURVEY.md §8d (this path moves no HBM
            bytes and has no GEMM: neither "hbm" nor "tensor" bounds it)
  cpu_baseline  the oracle port of the reference loop on this box's host cores (bounded sample; N=1 only)

BASELINE.json's metric has a second half and a second workload, carried as sub-records of the same line at every N:
  em         configs[2]: EM exact scheme, N=1000, 2^22 paths per GPU (weak): paths/s, ms_per_step, roofline, e2e
  c5_strong  configs[4]: FE and EM at 2^30 GLOBAL paths sharded over the N ranks (strong scaling), 3 steps each
  c4_sweep   configs[3]: the 20^3 (kappa, theta, sigma) grid with the reference's skip filter (7778 points), 2^20 GLOBAL
             paths per point sharded over the N ranks, ONE launch per method + one allreduce of 2 x 7778 moments
  other_floor (N=1)  configs[1] names both variance floors: the (.)+ floor on the headline workload, with the reference's
             CUDA build of that floor (its one floor token changed while compiling, oracle/_ref/nmch_ref_harness_plus)
             timed beside it and compared on the same seed
  group_check (N>1)  the single-process group front end (nmch_group_*: ncclCommInitAll, what the C++ classes and
             `--gpus` use) over the same N devices, run by rank 0 after the timed regions: its sums against the
             torch.distributed path's and its time per step

`--impl reference`: the reference arm.  The reference is a CUDA program with no CPU implementation; its hot
loop restated in C (oracle/, kind "port") is timed on ALL host threads this process may use, and when the
reference's own CUDA build (oracle/_ref/nmch_ref_harness) travelled to the box its measured throughput on
the same GPU is attached as "reference_cuda" -- that is the like-for-like number.
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
sys.path.insert(0, ROOT)

README = dict(T=1.0, S_0=1.0, v_0=0.1, r=0.0, k=0.5, rho=-0.7, theta=0.1, sigma=0.3)
HESTON_ANALYTIC = 0.1197325094                            # semi-analytic call at the README point (SURVEY.md §8c)
ISSUE_PER_CLK_PER_SM = min(128.0 / 42.0, 16.0 / 5.0)      # SURVEY.md §8d: 42 thread-instr, 5 MUFU per path-step
# Measured bounds of the kernels' OWN instruction mixes, issued from independent chains on a B200 SM sub-partition
# (profiles/microbench/pipe_rates2.cu -> profiles/r02_pipe_rates2.txt; cycles per warp-step per SMSP).  They are
# constants of a committed measurement ("static" below), not measured by this run.
MIX_BOUND_CYCLES_PER_WARP_STEP = 54.86                    # "FE mix, interleaved": 8 IMAD.WIDE, 11 ALU, 12 FP32, 4 MUFU
EM_MIX_BOUND_CYCLES_PER_WARP_TRIAL = 90.6                 # "r02 EM split, boosted, TWO trials" line / 2 (an estimate: the kernel overlaps its MUFUs better)
EM_TRIALS_PER_STEP = 1.045                                # Marsaglia-Tsang acceptance at the README point
# SURVEY.md §8d for EM: "estimate 90-100 instr/step => 3.9e8 paths/s/GPU ceiling at N=1000" = 95 thread-instr per
# path-step at one instruction per scheduler per clock
EM_INSTR_PER_PATH_STEP = 95.0
DUMP_LIMIT_BYTES = 64 << 20                               # --dump-outputs writes at most this much in all


# ------------------------------------------------------------------------------------------------
# clocks (NVML) sampled DURING the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self.power = [], set(), None, []
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    self.nv, "nvmlDeviceGetCurrentClocksEventReasons") else self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
                self.power.append(self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.nv:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._t:
            self._t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s), "power_w_max": max(self.power) if self.power else None}


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference's loop, all host threads, bounded sample
# ------------------------------------------------------------------------------------------------
def cpu_baseline(method: str, N: int, budget_s: float = 12.0):
    """value = units / (sample time - generator-initialisation time): the span the GPU arm's timed region covers
    (the reference reports curand_init separately as Tim_init, SURVEY.md §8d); init_s is measured on the same paths."""
    from oracle import oracle as o
    p = o.Params(N=N, **README)
    # NOT omp_get_max_threads(): torch.distributed.run exports OMP_NUM_THREADS=1 to every rank
    threads = o.host_threads()
    n = 1 << 13
    run = (lambda n: o.fe_run(p, rng=o.RNG_XORWOW, n_paths=n, threads=threads)) if method == "fe" else (
        lambda n: o.em_run(p, rng=o.RNG_XORWOW, n_paths=n, threads=threads))
    run(256)                                     # builds the skip-ahead tables outside the timed region
    t0 = time.perf_counter()
    run(n)
    dt = time.perf_counter() - t0
    while dt < min(1.0, budget_s) and n < (1 << 24):   # find the rate, then size one sample to the budget
        n *= 4
        t0 = time.perf_counter()
        run(n)
        dt = time.perf_counter() - t0
    n_big = int(min(max(n, n * budget_s / max(dt, 1e-9)), 1 << 26))
    n_big = max(1 << 13, 1 << (n_big.bit_length() - 1))
    t0 = time.perf_counter()
    run(n_big)
    dt = time.perf_counter() - t0
    t0 = time.perf_counter()
    o.rng_init_only(o.RNG_XORWOW, 1234, 0, n_big, threads)
    init_s = time.perf_counter() - t0
    loop_s = max(dt - init_s, 0.05 * dt)
    units = n_big * N if method == "fe" else n_big
    return {"value": units / loop_s, "unit": "path-steps/s" if method == "fe" else "paths/s", "cores": threads,
            "kind": "port", "init_s": init_s, "sample_s": dt, "value_incl_init": units / dt,
            "sample": f"{method.upper()} oracle (XORWOW stream), {n_big} paths x {N} steps on {threads} OpenMP threads: "
                      f"{dt:.2f} s in all, of which {init_s:.2f} s per-path curand_init (timed separately on the same "
                      f"paths and excluded from value, like the reference's Tim_init)"}


def _harness(method, rng, n, N, calls, kernel="k3", plus_floor=False):
    exe = os.path.join(ROOT, "oracle", "_ref", "nmch_ref_harness_plus" if plus_floor else "nmch_ref_harness")
    r = subprocess.run([exe, "--method", method, "--rng", rng, "--kernel", kernel, "--NTPB", "512", "--NB", str(n // 512),
                        "--N", str(N), "--repeat", str(calls)], capture_output=True, text=True, timeout=900, check=True)
    return [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]


def _var(row):
    return row["E2"] - row["E"] ** 2


def reference_cuda(method: str, log2_paths: int, N: int, repeat: int = 3, with_ours: bool = True, spread_runs: int = 5):
    """The reference's own CUDA build (unmodified sources, nvcc -arch=sm_100) on this GPU, if shipped.
    with_ours=False (the reference arm): only the reference binary runs -- nothing of this engine is loaded.
    The binary is run `spread_runs` times on the same seed: its float atomics make E and the variance differ from run
    to run, and that spread is what our same-seed differences have to be read against."""
    exe = os.path.join(ROOT, "oracle", "_ref", "nmch_ref_harness")
    if not os.path.exists(exe):
        return None
    try:
        import torch
        if not torch.cuda.is_available():
            return None
    except Exception:
        return None
    out = {}
    n = 1 << log2_paths
    units = n * N if method == "fe" else n
    for rng in ("xorwow", "philox"):
        try:
            runs = [_harness(method, rng, n, N, repeat + 1)[1:] for _ in range(max(1, spread_runs))]   # drop the warm-up call
            rows = runs[0]
            ms = min(x["exec_ms"] for run in runs for x in run)
            mean_E = [sum(run[c]["E"] for run in runs) / len(runs) for c in range(repeat)]
            mean_var = [sum(_var(run[c]) for run in runs) / len(runs) for c in range(repeat)]
            out[rng] = {"value": units / (ms * 1e-3), "exec_ms": ms, "init_ms": rows[0]["init_ms"],
                        "E": rows[-1]["E"], "E2": rows[-1]["E2"],
                        "own_spread": {"runs": len(runs),
                                       "max_rel_spread_E": max((max(r[c]["E"] for r in runs) - min(r[c]["E"] for r in runs))
                                                               / abs(mean_E[c]) for c in range(repeat)),
                                       "max_rel_spread_var": max((max(_var(r[c]) for r in runs) - min(_var(r[c]) for r in runs))
                                                                 / abs(mean_var[c]) for c in range(repeat)),
                                       "what": "same binary, same seed and calls, (max - min) / mean over the runs: "
                                               "the reference reduces with float atomics in arrival order"}}
            if not with_ours:
                continue

            kept = {}

            def same_seed(mode, tag):
                try:
                    from nmch_b200 import engine as E
                    with E.Engine(NTPB=512, NB=n // 512, N=N, method=E.METHOD_FE if method == "fe" else E.METHOD_EM,
                                  rng=mode, **README) as eng:
                        eng.init(1234)
                        eng.compute()
                        ours = [eng.compute() for _ in range(repeat)]
                    best = min(o_.exec_ms for o_ in ours)
                    kept[tag] = ours
                    out[rng][tag] = {
                        "value": units / (best * 1e-3), "exec_ms": best,
                        "max_rel_diff_E": max(abs(o_.mean - r_["E"]) / abs(r_["E"]) for o_, r_ in zip(ours, rows)),
                        "max_rel_diff_var": max(abs(o_.variance - _var(r_)) / _var(r_) for o_, r_ in zip(ours, rows)),
                        "max_rel_diff_E_vs_mean_of_runs": max(abs(o_.mean - m) / abs(m) for o_, m in zip(ours, mean_E)),
                        "max_rel_diff_var_vs_mean_of_runs": max(abs(o_.variance - m) / m for o_, m in zip(ours, mean_var))}
                except Exception as ex:  # noqa: BLE001
                    out[rng][tag] = {"error": str(ex)[:200]}

            from nmch_b200 import engine as E
            # same seed, same calls through OUR draw-compatible stream mode: identical draws, our timing
            same_seed(E.RNG_XORWOW_COMPAT if rng == "xorwow" else E.RNG_PHILOX_COMPAT, "ours_same_draws")
            if rng == "philox" and method == "fe":
                # the DEFAULT fast mode consumes the same Philox words and forms the same uniforms as the reference's
                # Philox instantiation: its own same-seed difference, at its own speed
                same_seed(E.RNG_PHILOX, "ours_native_same_words")
            if rng == "xorwow" and method == "fe":
                # the same integer draws through the native fast-math step (opt-in NMCH_RNG_XORWOW_FAST)
                same_seed(E.RNG_XORWOW_FAST, "ours_same_stream_fast")
                if "ours_same_draws" in kept and "ours_same_stream_fast" in kept:
                    a, b = kept["ours_same_draws"], kept["ours_same_stream_fast"]
                    out[rng]["fast_vs_compat"] = {
                        "max_rel_diff_E": max(abs(x.mean - y.mean) / abs(x.mean) for x, y in zip(a, b)),
                        "max_rel_diff_var": max(abs(x.variance - y.variance) / x.variance for x, y in zip(a, b)),
                        "what": "XORWOW_FAST against XORWOW_COMPAT on the same draws, both summed in FP64: the fast "
                                "transforms' own share of the differences above (what the two have in common against the "
                                "reference is the reference's FP32 accumulation, far above its run-to-run spread)"}
        except Exception as ex:  # noqa: BLE001
            out[rng] = {"error": str(ex)[:200]}
    out["what"] = (f"reference NMCH_{method.upper()}_K3_MM<rng> (unmodified sources, -O3 -arch=sm_100), 512 x {n // 512} "
                   f"paths, N={N}, best Tim_exec of {repeat} after one warm-up compute(), {spread_runs} runs of the binary; "
                   f"unit as `unit`")
    if with_ours:
        out["what"] += ("; ours_same_draws = this engine in the draw-compatible VALIDATION mode for that tag, same seed and "
                        "calls (a checker, not a performance mode: it runs the reference's IEEE transforms); "
                        "ours_same_stream_fast = the same XORWOW integer draws through the native fast-math step "
                        "(NMCH_RNG_XORWOW_FAST); ours_native_same_words (Philox tag) = the DEFAULT native mode, which "
                        "consumes the same Philox words and uniforms with fast transforms; max_rel_diff_* against run 1 of the reference and against the mean "
                        "of its runs, to be read against own_spread")
    return out


def reference_cuda_plus_floor(n: int, N: int, repeat: int = 3):
    """configs[1], the (.)+ side: the reference's CUDA build with its floor token `Vt = abs(Vt);` compiled as
    `Vt = fmaxf(Vt, 0.0f);` (oracle/Makefile: _ref/nmch_ref_harness_plus -- the reference codes only abs), and this
    engine on the same seed and calls: the draw-compatible mode of the tag and the fast mode on the same draws."""
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "nmch_ref_harness_plus")):
        return None
    from nmch_b200 import engine as E
    out = {"what": "reference NMCH_FE_K3_MM<rng> with the floor token changed to (.)+ while compiling (-O3 -arch=sm_100), "
                   f"512 x {n // 512} paths, N={N}, best Tim_exec of {repeat} after one warm-up compute(); ours on the same "
                   "seed and calls with floor = plus: max relative difference of E and of the variance"}
    for rng, modes in (("xorwow", (("ours_same_draws", E.RNG_XORWOW_COMPAT), ("ours_same_stream_fast", E.RNG_XORWOW_FAST))),
                       ("philox", (("ours_same_draws", E.RNG_PHILOX_COMPAT), ("ours_native_same_words", E.RNG_PHILOX)))):
        try:
            rows = _harness("fe", rng, n, N, repeat + 1, plus_floor=True)[1:]
            ms = min(x["exec_ms"] for x in rows)
            out[rng] = {"value": n * N / (ms * 1e-3), "exec_ms": ms, "E": rows[-1]["E"], "E2": rows[-1]["E2"]}
            for tag, mode in modes:
                with E.Engine(NTPB=512, NB=n // 512, N=N, rng=mode, floor=E.FLOOR_PLUS, **README) as eng:
                    eng.init(1234)
                    eng.compute()
                    ours = [eng.compute() for _ in range(repeat)]
                best = min(o_.exec_ms for o_ in ours)
                out[rng][tag] = {"value": n * N / (best * 1e-3), "exec_ms": best,
                                 "max_rel_diff_E": max(abs(o_.mean - r_["E"]) / abs(r_["E"]) for o_, r_ in zip(ours, rows)),
                                 "max_rel_diff_var": max(abs(o_.variance - _var(r_)) / _var(r_) for o_, r_ in zip(ours, rows))}
        except Exception as ex:  # noqa: BLE001
            out[rng] = {"error": str(ex)[:200]}
    return out


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline and of the em sub-record; c5_strong times a fixed 3 (2^30 paths per "
                         "step), c4_sweep one launch, other_floor / dense_mode / xorwow_fast_mode the best of 3")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--method", default="fe", choices=["fe", "em"])
    ap.add_argument("--log2-paths", type=int, default=None, help="paths per GPU (default 24 for FE, 22 for EM)")
    ap.add_argument("--N", type=int, default=1000)
    ap.add_argument("--floor", default="abs", choices=["abs", "plus"])
    ap.add_argument("--rng", default="philox", choices=["philox", "dense"],
                    help="philox: word-compatible native stream (default); dense: opt-in 3-steps-per-block FE stream")
    ap.add_argument("--paths-per-thread", type=int, default=0)
    ap.add_argument("--block-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-cuda", action="store_true")
    ap.add_argument("--no-sub-records", action="store_true", help="skip the em / c5_strong / group_check sub-records")
    ap.add_argument("--c5-log2-paths", type=int, default=30, help="GLOBAL paths of the c5_strong sub-record")
    ap.add_argument("--c4-log2-paths", type=int, default=20, help="GLOBAL paths per grid point of the c4_sweep sub-record")
    ap.add_argument("--c4-points", type=int, default=20, help="grid points per axis of the c4_sweep sub-record")
    ap.add_argument("--cpu-budget-s", type=float, default=None, help="seconds of host work per CPU-baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what each timed path returned in its last timed step as DIR/<name>.npy (FP64 moment sums)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU paths' results: it needs --impl ours")
    # the c4 arrays (16 bytes per grid point and method, at most c4_points^3 points) are the only ones that grow
    if args.dump_outputs and not args.no_sub_records and 2 * 16 * args.c4_points ** 3 > DUMP_LIMIT_BYTES - 1024:
        ap.error(f"--dump-outputs: --c4-points {args.c4_points} would write more than {DUMP_LIMIT_BYTES >> 20} MB")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    log2_paths = args.log2_paths if args.log2_paths is not None else (24 if args.method == "fe" else 22)
    n_per_gpu = 1 << log2_paths
    N = args.N

    def names(method):
        return (("fe_path_steps_per_s", "path-steps/s") if method == "fe" else ("em_paths_per_s", "paths/s"))

    metric, unit = names(args.method)
    workload = (f"BASELINE configs[1]: FE Euler |.| floor, README params, N={N}, 2^{log2_paths} paths per GPU, seed 1234"
                if args.method == "fe" else
                f"BASELINE configs[2]: EM exact scheme, README params, N={N}, 2^{log2_paths} paths per GPU, seed 1234")
    config = {"workload": workload, "method": args.method, "floor": args.floor, "rng": args.rng, "n_steps": N,
              "paths_per_gpu": n_per_gpu, "global_paths": n_per_gpu * world, "parallelism": f"paths sharded x{world}",
              "l2": "n/a: the kernel has no HBM-resident inputs (11 scalars by value), state lives in registers"}

    # ---------------------------------------------------------------- reference arm (host CPU port)
    if args.impl == "reference":
        if rank != 0:
            return 0
        times, walls = [], []
        base = None
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            base = cpu_baseline(args.method, N, budget_s=args.cpu_budget_s if args.cpu_budget_s is not None
                                else max(2.0, 60.0 / max(1, args.steps + args.warmup)))
            if i >= args.warmup:
                times.append(base["value"])
                walls.append(time.perf_counter() - t0)
        v = sum(times) / len(times)
        base["value"] = v
        line = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * sum(walls) / len(walls), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "cpu_baseline": base,
                "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "edo01/NMCH is CUDA-only; its hot loop restated in C (oracle/) is what runs on the host cores. "
                        "A rate of one host, whatever N: the GPU arm's value grows with N, so the ratio does too"}
        if not args.no_reference_cuda:
            line["reference_cuda"] = reference_cuda(args.method, log2_paths, N, with_ours=False)
        print(json.dumps(line))
        return 0

    # ---------------------------------------------------------------- our arm
    import torch
    import torch.distributed as dist

    from nmch_b200 import engine as E

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    saved_stdout = None
    host_group = None
    if world > 1:
        # NCCL prints its version banner on the C-level stdout when the communicator comes up: park fd 1 on stderr
        # until the JSON line is due, so that stdout carries exactly one line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
        # a HOST-side barrier for the group check: ranks must not wait in a spinning NCCL kernel on GPUs that rank 0
        # is about to drive from its own process
        host_group = dist.new_group(backend="gloo")

    from nmch_b200.distributed import ShardedEngine
    stream = torch.cuda.Stream(dev)             # one stream carries the kernel and the allreduce
    torch.cuda.set_stream(stream)

    # name -> what a timed path returned in its last timed step (FP64 moment sums), for --dump-outputs
    outputs = {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def measure(method, n_global, steps, warmup, rng=E.RNG_PHILOX, want_e2e=True, sample_clocks=False):
        """W untimed + exactly K timed compute() passes of `method` over n_global paths sharded over the ranks,
        CUDA events on the launching stream, max over ranks.  Returns a dict; the engine is closed on return."""
        sh = ShardedEngine(rank=rank, world=world, device=local_rank, NTPB=512, NB=n_global // 512, N=N,
                           method=E.METHOD_FE if method == "fe" else E.METHOD_EM,
                           floor=E.FLOOR_ABS if args.floor == "abs" else E.FLOOR_PLUS, rng=rng,
                           paths_per_thread=args.paths_per_thread if method == "fe" else 0,
                           block_threads=args.block_threads if method == "fe" else 0, **README)
        sh.init(1234)
        eng = sh.engine
        first = None
        moments = None
        for i in range(warmup):
            moments = sh.compute_async()             # kernel -> (N>1: one NCCL allreduce of 16 bytes of FP64 moments)
            if i == 0:
                first = moments.clone()
        barrier()
        launches0 = eng.launch_info()["kernel_launches"]
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(local_rank) as clocks:
            ev0.record(stream)
            for _ in range(steps):
                moments = sh.compute_async()
            ev1.record(stream)
            barrier()
        total_ms = max_over_ranks(ev0.elapsed_time(ev1))
        launches = eng.launch_info()["kernel_launches"] - launches0
        result = moments.cpu().numpy()
        first = first.cpu().numpy() if first is not None else None
        units_step = n_global * N if method == "fe" else n_global
        out = {"ms_per_step": total_ms / steps, "value": units_step / (total_ms / steps * 1e-3), "launches": int(launches),
               "result": result, "first": first, "info": eng.launch_info(), "clocks": clocks.summary() if sample_clocks else None,
               "n_local": eng.n_local}
        if want_e2e:
            # end to end through the public C-ABI call (host in, host out), every step
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                if world == 1:
                    eng.compute()                    # nmch_engine_compute: param upload + launch + sync + host result
                else:
                    sh.compute_async().cpu()         # D2H read of the reduced moments
            barrier()
            e2e_s = max_over_ranks(time.perf_counter() - t0)
            out["e2e"] = {"value": units_step * steps / e2e_s, "unit": names(method)[1],
                          "h2d_bytes_per_step": out["info"]["kernel_param_bytes"], "d2h_bytes_per_step": 16,
                          "api": "nmch_engine_compute (C ABI)" if world == 1 else "nmch_engine_compute_async + NCCL allreduce + D2H"}
        sh.close()
        return out

    def sweep(method, n_global, points_per_axis):
        """BASELINE configs[3]: the (kappa, theta, sigma) grid of src/NMCH/test/exploration.cu:46-52 at `points_per_axis`
        points per axis (computed in double, then cast), the reference's skip filter 20 k theta < sigma^2 applied
        (exploration.cu:76), every point on n_global paths sharded over the ranks: ONE launch + ONE allreduce."""
        import numpy as np
        P = points_per_axis
        ax = lambda lo, hi: [np.float32(lo + i * (hi - lo) / (P - 1)) if P > 1 else np.float32(lo) for i in range(P)]  # noqa: E731
        pts = [(k_, t_, s_) for s_ in ax(0.1, 1.0) for t_ in ax(0.01, 0.5) for k_ in ax(0.1, 10.0)
               if not (np.float32(20) * k_ * t_ < s_ * s_)]
        k_, t_, s_ = (np.array(x, np.float32) for x in zip(*pts))
        sh = ShardedEngine(rank=rank, world=world, device=local_rank, NTPB=512, NB=n_global // 512, N=N,
                           method=E.METHOD_FE if method == "fe" else E.METHOD_EM, rng=E.RNG_PHILOX, **README)
        sh.init(1234)
        sh.explore(k_[:4], t_[:4], s_[:4])                       # warm-up (also sizes nothing: buffers grow below)
        buf = sh._buffer(len(k_))
        barrier()
        l0 = sh.engine.launch_info()["kernel_launches"]
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        sh.engine.explore_async(stream.cuda_stream, k_, t_, s_, buf.data_ptr())
        from nmch_b200.distributed import allreduce_moments
        allreduce_moments(buf, None)
        ev1.record(stream)
        barrier()
        ms = max_over_ranks(ev0.elapsed_time(ev1))
        launches = sh.engine.launch_info()["kernel_launches"] - l0
        sums = buf.cpu().numpy().reshape(-1, 2)
        sh.close()
        outputs[f"c4_{method}_moments"] = sums
        means = sums[:, 0] / n_global
        units = len(k_) * n_global * (N if method == "fe" else 1)
        i0 = int(np.argmin(np.abs(k_ - 0.5) + np.abs(t_ - 0.1) * 10 + np.abs(s_ - 0.3) * 3))
        return {"points": len(k_), "paths_per_point": n_global, "launch_ms": ms, "gpu_launches": int(launches),
                "value": units / (ms * 1e-3), "unit": names(method)[1],
                "all_finite": bool(np.isfinite(sums).all()), "mean_of_E[X]": float(means.mean()),
                "nearest_to_README_point": {"k": float(k_[i0]), "theta": float(t_[i0]), "sigma": float(s_[i0]), "E[X]": float(means[i0])}}

    def stats(result, n_total):
        mean = float(result[0]) / n_total
        var = float(result[1]) / n_total - mean * mean
        return {"E[X]": mean, "var": var, "std_error": (max(var, 0.0) / n_total) ** 0.5, "heston_semi_analytic": HESTON_ANALYTIC}

    def roofline(method, per_gpu, info, f_mhz, f_max_mhz, dense=False):
        f_hz = (f_mhz or 1965) * 1e6
        sms = info["sm_count"]
        if method == "fe":
            peak = sms * f_hz * ISSUE_PER_CLK_PER_SM
            mix_peak = sms * f_hz * 4 * 32 / MIX_BOUND_CYCLES_PER_WARP_STEP
            model = ("SURVEY.md §8d: SMs x f x min(128/42 issue, 16/5 MUFU) path-steps/s; f = median SM clock sampled "
                     "during the timed region; per-GPU achieved")
        else:
            peak = sms * f_hz * 128.0 / (EM_INSTR_PER_PATH_STEP * N)
            mix_peak = sms * f_hz * 4 * 32 / (EM_MIX_BOUND_CYCLES_PER_WARP_TRIAL * EM_TRIALS_PER_STEP * N)
            model = ("SURVEY.md §8d estimate for EM: SMs x f x 128 / (95 thread-instr per path-step x N) paths/s "
                     "(data-dependent scheme: reported, not targeted; the round-2 sampler needs fewer instructions than "
                     "that estimate, so frac can exceed 1); f as for FE; per-GPU achieved")
        traffic = None
        tj = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tj):
            try:
                traffic = json.load(open(tj)).get("fe_dense" if (method == "fe" and dense) else method)
            except Exception:
                traffic = None
        return {"bound": "issue", "achieved": per_gpu, "peak": peak, "unit": names(method)[1], "frac": per_gpu / peak,
                "traffic": traffic,
                "traffic_source": "static: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed "
                                  "ncu --set full capture (profiles/traffic.json names it); not measured by this run. "
                                  "Algorithmic HBM bytes per launch: 0 (16 bytes of moments out)",
                "model": model,
                "peak_at_max_clock": sms * (f_max_mhz or 1965) * 1e6 * ISSUE_PER_CLK_PER_SM if method == "fe" else None,
                "mix_bound_peak": mix_peak, "mix_bound_frac": per_gpu / mix_peak,
                "mix_bound_source": "static: cycles per warp-step of the kernel's own instruction mix from independent "
                                    "chains, profiles/r02_pipe_rates2.txt (profiles/microbench/pipe_rates2.cu)"}

    # ---- headline
    head_rng = E.RNG_PHILOX_DENSE if (args.rng == "dense" and args.method == "fe") else E.RNG_PHILOX
    head = measure(args.method, n_per_gpu * world, args.steps, args.warmup, rng=head_rng, sample_clocks=True)
    assert head["n_local"] == n_per_gpu
    outputs["moments"] = head["result"]

    # ---- sub-records (every N): the EM half of BASELINE.json's metric, and configs[4] as strong scaling
    sub = {}
    if not args.no_sub_records and args.method == "fe" and args.rng == "philox":
        em = measure("em", (1 << 22) * world, args.steps, 3, sample_clocks=True)
        sub["em"] = em
        outputs["em_moments"] = em["result"]
        c5_n = 1 << args.c5_log2_paths
        c5 = {}
        for m in ("fe", "em"):
            c5[m] = measure(m, c5_n, 3, 1, want_e2e=False)
            outputs[f"c5_{m}_moments"] = c5[m]["result"]
        sub["c5"] = (c5_n, c5)
        sub["c4"] = {m: sweep(m, 1 << args.c4_log2_paths, args.c4_points) for m in ("fe", "em")}

    # ---- single-process group over the same devices (rank 0, everyone else parked on the host)
    group_check = None
    if world > 1 and not args.no_sub_records:
        torch.cuda.synchronize(dev)
        dist.barrier(group=host_group)               # every rank's GPU work is done; nobody spins on a device from here
        if rank == 0:
            try:
                with E.Group(world, NTPB=512, NB=(n_per_gpu * world) // 512, N=N,
                             method=E.METHOD_FE if args.method == "fe" else E.METHOD_EM, rng=head_rng,
                             floor=E.FLOOR_ABS if args.floor == "abs" else E.FLOOR_PLUS, **README) as g:
                    g.init(1234)
                    g_first = g.compute()            # call 1 after init == the torch path's first warm-up step
                    g.compute()
                    g_ms = [g.compute().exec_ms for _ in range(3)]
                t_first = head["first"]
                rel = max(abs(g_first.sum_payoff - t_first[0]) / abs(t_first[0]),
                          abs(g_first.sum_payoff_sq - t_first[1]) / abs(t_first[1]))
                group_check = {"n_gpus": world, "ms_per_step": sum(g_ms) / len(g_ms), "ms_per_step_min": min(g_ms),
                               "torch_path_ms_per_step": head["ms_per_step"],
                               "rel_ms_vs_torch_path": sum(g_ms) / len(g_ms) / head["ms_per_step"] - 1.0,
                               "sums_equal_torch_path": bool(g_first.sum_payoff == float(t_first[0]) and
                                                             g_first.sum_payoff_sq == float(t_first[1])),
                               "max_rel_diff_sums": rel,
                               "what": "nmch_group_* (one process, ncclCommInitAll over all N devices), same seed, same "
                                       "shards: first compute() after init against the torch.distributed path's first "
                                       "step; exec_ms = slowest device's event span incl. the allreduce, 3 steps"}
            except Exception as ex:  # noqa: BLE001
                group_check = {"error": str(ex)[:300]}
            torch.cuda.set_device(local_rank)
        dist.barrier(group=host_group)

    if saved_stdout is not None:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if rank == 0:
        info = head["info"]
        ck = head["clocks"]
        n_total = n_per_gpu * world
        per_gpu = head["value"] / world
        line = {
            "metric": metric, "value": head["value"], "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config,
            "e2e": head["e2e"],
            "gpu_launches": head["launches"],
            "clocks": ck,
            "roofline": roofline(args.method, per_gpu, info, ck["sm_mhz"], ck["sm_max_mhz"], dense=args.rng == "dense"),
            "kernel": {k: info[k] for k in ("grid_x", "grid_y", "block_threads", "paths_per_thread", "regs_per_thread", "sm_count")},
            "result": stats(head["result"], n_total),
        }
        if "em" in sub:
            em = sub["em"]
            eck = em["clocks"]
            line["em"] = {
                "metric": "em_paths_per_s", "value": em["value"], "unit": "paths/s", "ms_per_step": em["ms_per_step"],
                "steps": args.steps, "warmup": 3, "scaling": "weak", "gpu_launches": em["launches"],
                "config": {"workload": f"BASELINE configs[2]: EM exact scheme, README params, N={N}, 2^22 paths per GPU, seed 1234",
                           "paths_per_gpu": 1 << 22, "global_paths": (1 << 22) * world},
                "e2e": em["e2e"], "clocks": eck,
                "roofline": roofline("em", em["value"] / world, em["info"], eck["sm_mhz"], eck["sm_max_mhz"]),
                "kernel": {k: em["info"][k] for k in ("grid_x", "grid_y", "block_threads", "regs_per_thread")},
                "result": stats(em["result"], (1 << 22) * world)}
        if "c5" in sub:
            c5_n, c5 = sub["c5"]
            line["c5_strong"] = {
                "workload": f"BASELINE configs[4]: FE + EM at 2^{args.c5_log2_paths} GLOBAL paths, N={N}, sharded over "
                            f"{world} rank(s) with one NCCL moment allreduce per step", "scaling": "strong",
                "global_paths": c5_n, "steps": 3, "warmup": 1,
                "fe": {"ms_per_step": c5["fe"]["ms_per_step"], "value": c5["fe"]["value"], "unit": "path-steps/s",
                       "gpu_launches": c5["fe"]["launches"], "result": stats(c5["fe"]["result"], c5_n)},
                "em": {"ms_per_step": c5["em"]["ms_per_step"], "value": c5["em"]["value"], "unit": "paths/s",
                       "gpu_launches": c5["em"]["launches"], "result": stats(c5["em"]["result"], c5_n)}}
        if "c4" in sub:
            line["c4_sweep"] = {"workload": f"BASELINE configs[3]: {args.c4_points}^3 grid over kappa in [0.1,10], theta in [0.01,0.5], "
                                            f"sigma in [0.1,1] with the reference's skip filter, 2^{args.c4_log2_paths} GLOBAL paths per "
                                            f"point, N={N}, one launch per method, sharded over {world} rank(s)",
                                "scaling": "strong", "fe": sub["c4"]["fe"], "em": sub["c4"]["em"]}
        if group_check is not None:
            line["group_check"] = group_check
        if world == 1 and args.method == "fe" and args.rng == "philox" and not args.no_sub_records:
            peak = line["roofline"]["peak"]
            units_per_gpu_step = n_per_gpu * N
            try:                                  # configs[1] names both floors: the other one, same workload
                other = E.FLOOR_PLUS if args.floor == "abs" else E.FLOOR_ABS
                with E.Engine(NTPB=512, NB=n_per_gpu // 512, N=N, rng=E.RNG_PHILOX, device=local_rank, floor=other, **README) as fe2:
                    fe2.init(1234)
                    fe2.compute()
                    runs = [fe2.compute() for _ in range(3)]
                fms = min(r_.exec_ms for r_ in runs)
                line["other_floor"] = {"floor": "plus" if args.floor == "abs" else "abs", "value": units_per_gpu_step / (fms * 1e-3),
                                       "unit": unit, "ms_per_step": fms, "roofline_frac": units_per_gpu_step / (fms * 1e-3) / peak,
                                       "E[X]": runs[-1].mean, "std_error": runs[-1].std_error,
                                       "note": "BASELINE configs[1] is FE with the |.| floor vs the (.)+ floor: the headline is "
                                               "the reference's floor (|.|, the only one it codes), this is the other"}
                if other == E.FLOOR_PLUS and not args.no_reference_cuda:
                    line["other_floor"]["reference_cuda"] = reference_cuda_plus_floor(n_per_gpu, N)
            except Exception as ex:  # noqa: BLE001
                line["other_floor"] = {"error": str(ex)[:200]}
            try:                                  # the opt-in dense-draw stream, same workload, for the record
                with E.Engine(NTPB=512, NB=n_per_gpu // 512, N=N, rng=E.RNG_PHILOX_DENSE, device=local_rank,
                              floor=E.FLOOR_ABS if args.floor == "abs" else E.FLOOR_PLUS, **README) as de:
                    de.init(1234)
                    de.compute()
                    dms = min(de.compute().exec_ms for _ in range(3))
                dval = units_per_gpu_step / (dms * 1e-3)
                line["dense_mode"] = {"value": dval, "unit": unit, "ms_per_step": dms, "roofline_frac": dval / peak,
                                      "note": "NMCH_RNG_PHILOX_DENSE: three (23-bit, 19-bit) draws per Philox block; "
                                              "statistically equivalent, not cuRAND-word-compatible; bench.py --rng dense"}
            except Exception as ex:  # noqa: BLE001
                line["dense_mode"] = {"error": str(ex)[:200]}
            try:                                  # the reference's default stream (XORWOW) through the native step
                with E.Engine(NTPB=512, NB=n_per_gpu // 512, N=N, rng=E.RNG_XORWOW_FAST, device=local_rank,
                              floor=E.FLOOR_ABS if args.floor == "abs" else E.FLOOR_PLUS, **README) as xe:
                    xe.init(1234)
                    xe.compute()
                    xms = min(xe.compute().exec_ms for _ in range(3))
                    xinit = xe.init_ms
                xval = units_per_gpu_step / (xms * 1e-3)
                line["xorwow_fast_mode"] = {"value": xval, "unit": unit, "ms_per_step": xms, "init_ms": xinit,
                                            "note": "NMCH_RNG_XORWOW_FAST: cuRAND-XORWOW integer draws (the reference's "
                                                    "default generator, 24 B of state per path) through the native "
                                                    "fast-math step; same-seed agreement with the reference CUDA build "
                                                    "under reference_cuda.xorwow.ours_same_stream_fast"}
            except Exception as ex:  # noqa: BLE001
                line["xorwow_fast_mode"] = {"error": str(ex)[:200]}
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(args.method, N, budget_s=args.cpu_budget_s or 12.0)
        if not args.no_reference_cuda and world == 1:
            line["reference_cuda"] = reference_cuda(args.method, log2_paths, N)
            if "em" in line:
                line["em"]["reference_cuda"] = reference_cuda("em", 22, N, spread_runs=2)
        if args.dump_outputs:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in outputs.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), np.asarray(arr, dtype=np.float64))
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
