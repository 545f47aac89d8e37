"""Times compute_sensitivities() against the passes it builds on, in one run on one GPU (DESIGN.md §4.6c).

Setup: 2^24 paths x 1000 steps at the README point (T = 1, S_0 = 1, v_0 = 0.1, r = 0, k = 0.5, rho = -0.7, theta = 0.1,
sigma = 0.3), both floors, 1 and 64 strikes.  Per setup, after a warm-up of every call, `--reps` rounds each of:
compute(), compute_strikes(), compute_greeks(), compute_sensitivities(), six compute_strikes() passes (the one-sided
bump-and-revalue that the sensitivities replace) and compute_greeks() of a separately built library of the parent commit
(--parent-lib, same C ABI), alternated round by round.  Times are the engines' device-event spans (exec_ms).  A separate
torch.profiler window splits compute_sensitivities() into its tangent kernel and its fold.  Also records registers per
thread, the GPU name and its power limit.  --variant-lib times compute_sensitivities() of another build of this library
(e.g. one path per thread, NMCHB_SENS_PATHS=1).

    python scripts/sensitivities_time.py --parent-lib nmch_b200/variants/parent/libnmch_b200_parent.so \\
        --out profiles/r03_sensitivities_time.json
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from nmch_b200 import capi  # noqa: E402
from nmch_b200 import engine as E  # noqa: E402

README = dict(T=1.0, S_0=1.0, v_0=0.1, r=0.0, k=0.5, rho=-0.7, theta=0.1, sigma=0.3)


class RawEngine:
    """An engine of another build of the same C ABI (loaded by path), for the calls this script times."""

    def __init__(self, path, **kw):
        self.L = C.CDLL(path)
        vp = C.c_void_p
        self.L.nmch_engine_create.argtypes = [C.POINTER(capi.NmchParams), C.POINTER(vp)]
        self.L.nmch_engine_init.argtypes = [vp, C.c_ulonglong]
        self.L.nmch_engine_compute_greeks.argtypes = [vp, C.POINTER(C.c_float), C.c_int, C.POINTER(capi.NmchGreekMoments)]
        self.L.nmch_engine_destroy.argtypes = [vp]
        self.L.nmch_engine_destroy.restype = None
        self.has_sens = hasattr(self.L, "nmch_engine_compute_sensitivities")
        if self.has_sens:
            self.L.nmch_engine_compute_sensitivities.argtypes = [vp, C.POINTER(C.c_float), C.c_int,
                                                                 C.POINTER(capi.NmchSensitivityMoments)]
        d = dict(NTPB=512, NB=512, T=1.0, S_0=1.0, v_0=0.1, r=0.0, k=0.5, rho=-0.7, theta=0.1, sigma=0.3, N=1000,
                 method=0, floor=0, rng=0, device=-1, n_paths=0, first_path=0, n_local=0, paths_per_thread=0,
                 block_threads=0)
        d.update(kw)
        self.p = capi.NmchParams(*[d[n] for n, _ in capi.NmchParams._fields_])
        self.h = C.c_void_p()
        assert self.L.nmch_engine_create(C.byref(self.p), C.byref(self.h)) == 0

    def init(self, seed):
        assert self.L.nmch_engine_init(self.h, seed) == 0

    def greeks_ms(self, strikes):
        out = (capi.NmchGreekMoments * len(strikes))()
        assert self.L.nmch_engine_compute_greeks(self.h, strikes.ctypes.data_as(C.POINTER(C.c_float)), len(strikes), out) == 0
        return out[0].exec_ms

    def sens_ms(self, strikes):
        out = (capi.NmchSensitivityMoments * len(strikes))()
        assert self.L.nmch_engine_compute_sensitivities(self.h, strikes.ctypes.data_as(C.POINTER(C.c_float)),
                                                        len(strikes), out) == 0
        return out[0].exec_ms

    def close(self):
        self.L.nmch_engine_destroy(self.h)


def gpu_facts():
    import torch
    facts = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        facts["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0]
    except Exception as exc:          # the numbers stay valid; the record says why the limit is missing
        facts["power_limit_and_max_sm_clock"] = f"not read: {exc}"
    return facts


def kernel_split(e, strikes, reps):
    """Device time per kernel name over `reps` compute_sensitivities() calls, from torch.profiler (a window of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            e.compute_sensitivities(strikes)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name != "CUDA" or ev.count == 0:
            continue
        name = ev.key
        tag = "tangent_kernel" if "fe_tangent_kernel" in name else "fold" if "strike_fold_kernel" in name else None
        if tag:
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            out[tag] = {"name": name[:120], "ms_per_call": t / 1e3 / reps, "calls": ev.count}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True)
    ap.add_argument("--variant-lib", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_sensitivities_time.json"))
    ap.add_argument("--log2-paths", type=int, default=24)
    ap.add_argument("--N", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    n = 1 << a.log2_paths
    rec = {"setup": dict(README, n_paths=n, N=a.N, reps=a.reps, unit="ms, device events (exec_ms), median of reps"),
           **gpu_facts(), "rows": []}
    for floor in (0, 1):
        for n_strikes in (1, 64):
            strikes = np.ascontiguousarray(np.linspace(0.7, 1.3, n_strikes) if n_strikes > 1 else [1.0], np.float32)
            kw = dict(README, NTPB=512, NB=n // 512, N=a.N, floor=floor)
            e = E.Engine(**kw).init(1234)
            par = RawEngine(a.parent_lib, **kw)
            par.init(1234)
            var = None
            if a.variant_lib:
                var = RawEngine(a.variant_lib, **kw)
                var.init(1234)
            calls = {
                "compute": lambda: e.compute().exec_ms,
                "compute_strikes": lambda: e.compute_strikes(strikes)[0]["moments"].exec_ms,
                "compute_greeks": lambda: e.compute_greeks(strikes)[0]["moments"].exec_ms,
                "compute_greeks_parent": lambda: par.greeks_ms(strikes),
                "compute_sensitivities": lambda: e.compute_sensitivities(strikes)[0]["moments"].exec_ms,
                "six_compute_strikes": lambda: sum(e.compute_strikes(strikes)[0]["moments"].exec_ms for _ in range(6)),
            }
            if var is not None and var.has_sens:
                calls["compute_sensitivities_variant"] = lambda: var.sens_ms(strikes)
            for f in calls.values():                       # warm-up: module load, buffers, first launches
                f()
            times = {k: [] for k in calls}
            for _ in range(a.reps):
                for k, f in calls.items():
                    times[k].append(f())
            row = {"floor": "abs" if floor == 0 else "plus", "n_strikes": n_strikes}
            for k, v in times.items():
                row[k] = {"median": statistics.median(v), "min": min(v), "max": max(v)}
            row["sensitivities_over_six_strike_passes"] = row["compute_sensitivities"]["median"] / row["six_compute_strikes"]["median"]
            row["greeks_over_parent_greeks"] = row["compute_greeks"]["median"] / row["compute_greeks_parent"]["median"]
            e.compute_sensitivities(strikes)
            row["regs_sensitivities_tangent"] = e.launch_info()["regs_per_thread"]
            row["paths_per_thread_sensitivities"] = e.launch_info()["paths_per_thread"]
            e.compute_greeks(strikes)
            row["regs_greeks_tangent"] = e.launch_info()["regs_per_thread"]
            row["kernels_sensitivities"] = kernel_split(e, strikes, a.reps)
            print(json.dumps(row), flush=True)
            rec["rows"].append(row)
            e.close()
            par.close()
            if var is not None:
                var.close()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
