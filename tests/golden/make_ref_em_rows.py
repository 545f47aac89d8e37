#!/usr/bin/env python
"""Regenerates tests/golden/ref_em_rows.json from the reference's own CUDA build (oracle/_ref/nmch_ref_harness, built by
`make -C oracle ref REF=<reference checkout>`): the EM rows tests/ref_build.py returns when that build is absent.  It refuses
to run without the build.

The rows stored now were recorded from this engine's draw-compatible EM modes, on the engine and test sources of
profiles/r02_test_gpu_1gpu.txt.  That log has 272 GPU tests passed and 8 skipped.  The 8 skips are the two-device tests, so
every test that ran the reference build passed, including all the cases below at 1e-5 in price and variance.  Those sources
are unchanged since.  Where the reference's own EM output is stored (tests/golden/ref_cuda_b200.json) the rows agree with it
to 2e-7.  Rerun this script with the build to replace them with the build's own rows.

Run on a B200:   python tests/golden/make_ref_em_rows.py
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import ref_build  # noqa: E402
from oracle import oracle as o  # noqa: E402

# every EM harness call of tests/test_gpu_em.py and tests/test_cpp_api.py (K1 classes: live only, tests/ref_build.py)
CFG = [dict(NTPB=512, NB=64, N=1000), dict(NTPB=128, NB=32, N=250), dict(NTPB=512, NB=32, N=500, k=2.08, theta=0.108, sigma=1.0)]
SEED_CFG = [dict(NTPB=256, NB=64, N=200), dict(NTPB=256, NB=64, N=200, k=10.0, theta=0.5, sigma=1.0),
            dict(NTPB=256, NB=64, N=120, T=0.5, v_0=0.04, k=1.5, rho=0.3, theta=0.09, sigma=0.5)]
CASES = [dict(method="em", rng=r, kernel="k3", repeat=2, **c) for r in ("xorwow", "philox", "mrg") for c in CFG]
CASES += [dict(method="em", rng=r, kernel="k3", repeat=2, seed=s, **c)
          for s in (0, 0xFEDCBA9876543210) for r in ("xorwow", "philox", "mrg") for c in SEED_CFG]
CASES += [dict(method="em", rng=r, kernel=k, NTPB=128, NB=32, N=60, repeat=2) for k in ("k2", "k3") for r in ("xorwow", "mrg")]


def main():
    if not os.path.exists(o.REF_HARNESS_PATH):
        raise SystemExit(f"{o.REF_HARNESS_PATH} is missing: build it with `make -C oracle ref REF=<reference checkout>`")
    rows = {ref_build.key(c): ref_build.harness_rows(**c) for c in CASES}
    gold = {"generator": "oracle/_ref/nmch_ref_harness (reference sources) on a B200", "rows": rows}
    with open(os.path.join(HERE, "ref_em_rows.json"), "w") as f:
        json.dump(gold, f, indent=1)
    print("wrote", len(rows), "cases to", os.path.join(HERE, "ref_em_rows.json"))


if __name__ == "__main__":
    main()
