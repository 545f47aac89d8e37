"""What the reference's own CUDA build prints for a set of harness flags (oracle/_ref/nmch_ref_harness: one JSON row per
compute() call, with the float E[X], E[X^2] and err its getters return), for the tests that compare against it.

That build is compiled from a checkout of the reference (oracle/Makefile), which is not part of this repository.  When it
is present it runs live.  Without it the rows come from:
  * FE: the oracle (oracle/, the reference's FE loop restated in C on cuRAND's streams), which reproduces the reference
    build's stored outputs (tests/golden/ref_cuda_b200*.json, tests/test_ref_cuda_golden.py) to 3e-6 -- the comparisons
    ask for 1e-5;
  * EM: tests/golden/ref_em_rows.json (tests/golden/make_ref_em_rows.py).  The oracle's EM takes cuRAND's host branches,
    which flip rare accept / reject decisions, so it cannot stand in at 1e-5.
The K1 classes (--kernel k1 / k1pgm / k1pim) store E[X^2] / n^2 through their own reduction: only their build can show
what they return, so without it those comparisons skip.
"""
import json
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as o

EM_ROWS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_em_rows.json")
PKEYS = ("T", "S_0", "v_0", "r", "k", "rho", "theta", "sigma")
K1_KERNELS = ("k1", "k1pgm", "k1pim")
RNGS = {"xorwow": o.RNG_XORWOW, "philox": o.RNG_PHILOX, "mrg": o.RNG_MRG32K3A}
DEFAULTS = dict(method="fe", rng="xorwow", kernel="k3", NTPB=512, NB=512, N=1000, seed=1234, repeat=1)   # ref_harness.cu


def key(flags) -> str:
    """Flags as the harness reads them (every value a string), defaults filled in."""
    return json.dumps({k: str(v) for k, v in sorted({**DEFAULTS, **flags}.items())})


def ref_err(n: int, E: float, E2: float) -> float:
    """The reference's 95 % half-width from its float getters (NMCH_FE.hpp:50-55; nmch_b200/methods.py get_err)."""
    inner = float(np.float32(n) * np.float32(E2) - np.float32(E) * np.float32(E))
    if inner < 0:
        return float("nan")
    return float(np.float32(1.96 * math.sqrt(float(np.float32(1.0) / np.float32(n - 1)) * inner) / math.sqrt(float(n))))


def row(n: int, mean: float, mean_sq: float) -> dict:
    E, E2 = float(np.float32(mean)), float(np.float32(mean_sq))
    return {"E": E, "E2": E2, "err": ref_err(n, E, E2), "cuda": "cudaSuccess"}


def _oracle_fe(plus_floor: bool, flags: dict):
    f = {**DEFAULTS, **flags}
    n = int(f["NTPB"]) * int(f["NB"])
    p = o.Params(N=int(f["N"]), **{k: float(f[k]) for k in PKEYS if k in f})
    out = []
    for call in range(1, int(f["repeat"]) + 1):
        r = o.fe_run(p, rng=RNGS[f["rng"]], floor=o.FLOOR_PLUS if plus_floor else o.FLOOR_ABS, seed=int(f["seed"]),
                     n_paths=n, calls=call)
        out.append(row(n, r["mean"], r["mean_sq"]))
    return out


def harness_rows(plus_floor: bool = False, timeout: int = 900, **flags):
    """plus_floor: the reference build with its FE floor token changed to (.)+ (oracle/Makefile)."""
    exe = o.REF_HARNESS_PLUS_PATH if plus_floor else o.REF_HARNESS_PATH
    if os.path.exists(exe):
        cmd = [exe]
        for k, v in flags.items():
            cmd += [f"--{k}", str(v)]
        out = subprocess.run(cmd, check=True, capture_output=True, text=True, timeout=timeout).stdout
        # the reference's get_err() is NaN under its own K1 quirk and printf writes "-nan": not JSON
        return [json.loads(l.replace("-nan", "NaN").replace(" nan", " NaN")) for l in out.splitlines() if l.startswith("{")]
    if {**DEFAULTS, **flags}["kernel"] in K1_KERNELS:
        pytest.skip(f"{exe} is missing: the reference's K1 classes (E[X^2] / n^2) can only be compared with their build")
    if {**DEFAULTS, **flags}["method"] == "fe":
        return _oracle_fe(plus_floor, flags)
    assert not plus_floor, "the (.)+ floor exists in FE only"
    with open(EM_ROWS) as f:
        stored = json.load(f)["rows"]
    assert key(flags) in stored, f"no stored EM rows for {key(flags)}: add the case to tests/golden/make_ref_em_rows.py"
    return stored[key(flags)]
