"""The QE pass (qe_kernel) against the float64 QE-M reference (tests/qe64_reference.py) on the same Philox draws, at the
edges the path kernels are tested at: N = 1 and odd N, 64-bit seeds, ragged shards, first_path beyond 2^32 and shards
across it, r != 0, S_0 in {0.5, 100}, T != 1, rho from -0.9 to +0.9, the Feller-violating point, kappa = 10, theta = 0
(from v_0 > 0 and from v_0 = 0), theta in {1e-12, 1e-20} and sigma in {0.01, 1e-3}.  Per path (compute_paths), the
FP64 payoff sums of compute() and explore(), and compute_strikes() at K = 0 and quantile strikes, each at the call id
the engine's call counter should have reached."""
import ctypes as C

import numpy as np
import pytest

import fe64_reference as F
import qe64_reference as R

# Tolerances, each at most 10x the largest value measured over CONFIGS (NVIDIA B200, 1000 W power limit).
DELTA_S = 1e-4          # per-path relative error of S_T, the same at every sigma; measured 2.2e-6 at sigma = 0.3
                        # (configuration 11), 4.8e-7 at sigma = 1e-3 (configuration 10), 1.1e-5 at theta = 1e-20
                        # (configuration 8, most paths parked at V = 0).  The cancelling log-price form of the parent
                        # kernel measured 3.7e-4 at sigma = 1e-3.
RTOL_V = 5e-3           # per-path |V_T - V_ref| / (V_ref + 1e-2 mean V_ref); measured 5.8e-4 (theta = 0,
                        # configuration 5), 1.8e-5 elsewhere
RTOL_SUMS = 9e-5        # payoff, payoff^2, delta and itm sums of compute(), explore() and compute_strikes() outside
                        # the reference bounds, relative to the sum of |terms|; measured 3.4e-7 at K = 0, 9.2e-6 at the
                        # quantile strikes, 3.3e-6 for compute() and 2.1e-6 for explore()
# Not tolerances: paths that came within PSI_MARGIN of the psi = 1.5 switch (float32 and float64 may take different
# branches there, and V' jumps) or within U_MARGIN of the point mass of the exponential branch are left out of the
# per-path comparison; the share left out is bounded by MAX_LEFT_OUT, so the mask cannot hide a systematic error.
PSI_MARGIN, U_MARGIN = 1e-3, 1e-5
MAX_LEFT_OUT = 0.03     # measured 6.5e-3 (the Feller-violating configuration 3)
QUANTILES = [0.05, 0.2, 0.35, 0.5, 0.65, 0.8, 0.95]
PARAMS = ("T", "S_0", "v_0", "r", "k", "rho", "theta", "sigma")

EDGES = [dict(N=1), dict(rho=0.9, hi=1), dict(straddle=True), dict(k=2.08, theta=0.108, sigma=1.0),
         dict(k=10.0, theta=0.5, sigma=1.0, N=5), dict(theta=0.0, v_0=0.1), dict(theta=0.0, v_0=0.0), dict(theta=1e-12),
         dict(theta=1e-20, sigma=1.0, v_0=0.05, hi=1), dict(sigma=0.01, rho=-0.9), dict(sigma=1e-3, rho=-0.7, k=0.5, theta=0.1),
         dict(sigma=0.3, rho=-0.7, k=0.5, theta=0.1), dict(rho=-0.9, straddle=True)]


def _configs(seed):
    """One seeded random configuration per entry of EDGES, with the entry's values imposed.  The pass under test
    follows nothing, one compute() or a two-point explore() (call ids 0, 1, 2), in turn."""
    r = np.random.default_rng(seed)
    for i, edge in enumerate(EDGES):
        c = dict(T=float(r.choice([0.25, 0.5, 2.0])), S_0=float(r.choice([0.5, 1.0, 100.0])),
                 v_0=float(r.uniform(0.01, 0.3)), r=float(r.choice([0.0, 0.01, 0.05])), k=float(r.uniform(0.2, 6.0)),
                 rho=float(r.uniform(-0.9, 0.9)), theta=float(r.uniform(0.02, 0.4)), sigma=float(r.uniform(0.1, 0.9)),
                 N=int(r.integers(1, 60)) * 2 + (i % 2), n=int(r.integers(300, 4097)),
                 seed=int(r.integers(1, 2 ** 31)) << 32 | int(r.integers(0, 2 ** 32)),
                 first=int(r.integers(0, 50)) * 4096, advance=("none", "compute", "explore")[i % 3])
        c.update({k: v for k, v in edge.items() if k in c})
        if edge.get("hi"):
            c["first"] += 1 << 32                       # path_hi = 1
        if edge.get("straddle"):
            c["first"], c["n"] = (1 << 32) - 4096, 4096 + 1000
        yield c


CONFIGS = list(_configs(2026))


def _engine(c):
    from nmch_b200 import engine as E
    return E.Engine(NTPB=1, NB=1, N=c["N"], method=E.METHOD_QE, n_paths=c["first"] + c["n"], first_path=c["first"],
                    n_local=c["n"], **{p: c[p] for p in PARAMS})


def _ref(c, call, **over):
    kw = {p: c[p] for p in PARAMS}
    kw.update(over)
    return R.qe_paths(**kw, N=c["N"], seed=c["seed"], first_path=c["first"], n_paths=c["n"], call=call)


def _strike_sums(e, strikes):
    """compute_strikes' raw FP64 sums, shape (n_strikes, 4): payoff, payoff^2, delta, itm."""
    from nmch_b200 import capi
    strikes = np.ascontiguousarray(strikes, np.float32)
    out = (capi.NmchStrikeMoments * len(strikes))()
    capi.check(e._lib.nmch_engine_compute_strikes(e._h, strikes.ctypes.data_as(C.POINTER(C.c_float)), len(strikes), out))
    return np.array([[m.sum_payoff, m.sum_payoff_sq, m.sum_delta, m.sum_itm] for m in out])


def _outside(got, ref, K, S_0, nsums):
    """How far the first nsums sums of strike K lie outside the reference bounds, relative to the sum of |terms|."""
    lo, hi, scale = F.strike_fold_bounds(ref.S, np.zeros_like(ref.S), K, S_0, DELTA_S)
    lo, hi, scale = lo[:nsums], hi[:nsums], scale[:nsums]
    return float(np.max(np.maximum(np.maximum(lo - got, got - hi), 0.0) / np.maximum(scale, 1e-300)))


def measure_config(c):
    """Runs one configuration; returns what the assertions of test_qe_matches_the_float64_reference bound."""
    out = {}
    pts = ((c["k"], c["theta"], c["sigma"]), (1.5 * c["k"], 0.5 * c["theta"], 0.5 * c["sigma"]))
    with _engine(c) as e:
        e.init(c["seed"])
        call0 = 0
        if c["advance"] == "compute":
            e.compute()
            call0 = 1
        elif c["advance"] == "explore":
            ex = e.explore(*[[p[j] for p in pts] for j in range(3)])
            # point i runs with its own parameters and call id i
            out["explore"] = max(_outside(np.array([m.sum_payoff, m.sum_payoff_sq]),
                                          _ref(c, i, k=kk, theta=th, sigma=sg), c["S_0"], c["S_0"], 2)
                                 for i, (m, (kk, th, sg)) in enumerate(zip(ex, pts)))
            call0 = 2
        S, V, _ = e.compute_paths()
        ref = _ref(c, call0)
        ref1 = _ref(c, call0 + 1)
        got1 = _strike_sums(e, np.concatenate([[0.0], np.quantile(ref1.S, QUANTILES)]))
        m2 = e.compute()
    ok = (ref.psi_margin > PSI_MARGIN) & (ref.u_margin > U_MARGIN)
    out["left_out"] = float(1.0 - ok.mean())
    out["no_martingale"] = int(ref.no_martingale.sum())
    out["parked"] = float((ref.V == 0.0).mean())
    out["finite"] = bool(np.isfinite(S).all() and np.isfinite(V).all())
    out["S_path"] = float(np.max(np.abs(S[ok] / ref.S[ok] - 1.0)))
    out["V_path"] = float(np.max(np.abs(V[ok] - ref.V[ok]) / (ref.V[ok] + 1e-2 * ref.V.mean() + 1e-300)))
    out["k0"] = _outside(got1[0], ref1, 0.0, c["S_0"], 4)
    out["q"] = max(_outside(got1[j], ref1, K, c["S_0"], 4) for j, K in enumerate(np.quantile(ref1.S, QUANTILES), 1))
    out["compute"] = _outside(np.array([m2.sum_payoff, m2.sum_payoff_sq]), _ref(c, call0 + 2), c["S_0"], c["S_0"], 2)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(CONFIGS)))
def test_qe_matches_the_float64_reference(i):
    c = CONFIGS[i]
    m = measure_config(c)
    assert m["finite"] and m["no_martingale"] == 0, (m, c)
    assert m["left_out"] <= MAX_LEFT_OUT, (m, c)
    assert m["S_path"] < DELTA_S and m["V_path"] < RTOL_V, (m, c)
    assert m["k0"] < RTOL_SUMS and m["q"] < RTOL_SUMS, (m, c)
    assert m["compute"] < RTOL_SUMS and m.get("explore", 0.0) < RTOL_SUMS, (m, c)


def test_configurations_cover_the_edges():
    """The configurations reach what the module docstring promises (this checks the test, not the kernel)."""
    firsts = [(c["first"], c["first"] + c["n"]) for c in CONFIGS]
    assert any(a >= 1 << 32 for a, _ in firsts) and any(a < 1 << 32 < b for a, b in firsts)
    assert {c["advance"] for c in CONFIGS} == {"none", "compute", "explore"}
    assert any(c["N"] == 1 for c in CONFIGS) and any(c["N"] % 2 for c in CONFIGS)
    assert all(c["seed"] >> 32 for c in CONFIGS) and any(c["n"] % 256 for c in CONFIGS)
    assert min(c["rho"] for c in CONFIGS) <= -0.9 and max(c["rho"] for c in CONFIGS) >= 0.9
    assert {0.0, 1e-12, 1e-20} <= {c["theta"] for c in CONFIGS} and {0.01, 1e-3} <= {c["sigma"] for c in CONFIGS}
    assert any(c["theta"] == 0.0 and c["v_0"] == 0.0 for c in CONFIGS)
    assert any(c["theta"] == 0.0 and c["v_0"] > 0.0 for c in CONFIGS)
    assert {0.5, 100.0} <= {c["S_0"] for c in CONFIGS} and any(c["r"] for c in CONFIGS)
    # theta = 1e-20: some paths park at V = 0, where m^2 = (theta (1 - e^{-k dt}))^2 is below float32's normal range
    tiny = next(c for c in CONFIGS if c["theta"] == 1e-20)
    m0 = tiny["theta"] * -np.expm1(-tiny["k"] * tiny["T"] / tiny["N"])
    assert m0 * m0 < np.finfo(np.float32).tiny and (_ref(tiny, 2).V == 0.0).mean() > 0.05
