"""GPU parity tests of the EM ("exact method") hot path, through the C ABI.

Bars (BASELINE.json north_star; SURVEY.md §7 hard part 4):
  * compat modes reproduce the reference's draw sequence, so they must match the reference's CUDA build
    on identical seeds to 1e-5 relative on price and variance -- including its Poisson-sampler bias;
  * the native mode is statistically exact: within 3 SE of the semi-analytic Heston price and of the
    oracle's exact-sampler restatement of the same scheme, with E[S_T] = S_0 e^{rT} (martingale).
The CPU oracle's EM takes cuRAND's HOST branches (expf/logf instead of ex2/lg2.approx), so a rare
accept/reject decision differs between host and device: host-vs-device EM parity is per-path for the
overwhelming majority of paths and statistical in aggregate.
"""
import numpy as np
import pytest

from oracle import oracle as o
from ref_build import harness_rows

pytestmark = pytest.mark.gpu

E = None


@pytest.fixture(scope="module", autouse=True)
def _engine_module():
    global E
    from nmch_b200 import engine as _e
    E = _e
    yield


def em_engine(n, N=1000, rng=0, **kw):
    ntpb = min(n, 512)
    return E.Engine(NTPB=ntpb, NB=n // ntpb, N=N, method=E.METHOD_EM, rng=rng, **kw)


def em_engine_n(n, N, **kw):
    return E.Engine(NTPB=1, NB=1, N=N, method=E.METHOD_EM, n_paths=n, **kw)


def _ref_cuda(**flags):
    return harness_rows(timeout=900, **flags)


def _rel(a, b):
    return abs(a - b) / abs(b)


# ---------------------------------------------------------------------------------------------
# compat vs oracle and vs the reference CUDA build
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rng_e,rng_o", [(1, o.RNG_XORWOW), (2, o.RNG_PHILOX), (3, o.RNG_MRG32K3A)])
def test_compat_tracks_oracle(rng_e, rng_o):
    n, N = 2048, 100
    with em_engine(n, N, rng=rng_e) as e:
        e.init(1234)
        S, V, m = e.compute_paths()
    ref = o.em_run(o.Params(N=N), rng=rng_o, n_paths=n, want_paths=True)
    close = np.isclose(S, ref["S"], rtol=2e-3, atol=2e-4)
    assert close.mean() > 0.97, close.mean()               # a flipped accept/reject re-routes a path
    se = o.std_error(ref["mean"], ref["mean_sq"], n)
    assert abs(m.mean - ref["mean"]) < 0.5 * se


@pytest.mark.parametrize("rng_name,rng_e", [("xorwow", 1), ("philox", 2), ("mrg", 3)])
@pytest.mark.parametrize("cfg", [dict(NTPB=512, NB=64, N=1000), dict(NTPB=128, NB=32, N=250),
                                 dict(NTPB=512, NB=32, N=500, k=2.08, theta=0.108, sigma=1.0)])
def test_compat_matches_reference_cuda_build(rng_name, rng_e, cfg):
    ref = _ref_cuda(method="em", rng=rng_name, kernel="k3", repeat=2, **cfg)
    kw = {k: cfg[k] for k in ("k", "theta", "sigma") if k in cfg}
    with E.Engine(NTPB=cfg["NTPB"], NB=cfg["NB"], N=cfg["N"], method=E.METHOD_EM, rng=rng_e, **kw) as e:
        e.init(1234)
        for call in range(2):
            m = e.compute()
            r = ref[call]
            assert r["cuda"] == "cudaSuccess"
            assert _rel(m.mean, r["E"]) < 1e-5, (call, m.mean, r["E"])
            assert _rel(m.variance, r["E2"] - r["E"] ** 2) < 1e-5, (call, m.variance)


@pytest.mark.parametrize("seed", [0, 0xFEDCBA9876543210])
@pytest.mark.parametrize("rng_name,rng_e", [("xorwow", 1), ("philox", 2), ("mrg", 3)])
@pytest.mark.parametrize("cfg", [dict(NTPB=256, NB=64, N=200), dict(NTPB=256, NB=64, N=200, k=10.0, theta=0.5, sigma=1.0),
                                 dict(NTPB=256, NB=64, N=120, T=0.5, v_0=0.04, k=1.5, rho=0.3, theta=0.09, sigma=0.5)])
def test_compat_other_seeds_and_parameters_match_the_reference_cuda_build(seed, rng_name, rng_e, cfg):
    """Other seeds (zero; 64 bits with a non-zero high half) and parameter sets (large shape and noncentrality; T != 1 with the
    reference's own T = 1 formula for the terminal draw, NMCH_EM.cu:116): the draw-compatible mode follows every accept /
    reject decision of the reference's cuRAND samplers."""
    ref = _ref_cuda(method="em", rng=rng_name, kernel="k3", repeat=2, seed=seed, **cfg)
    kw = {k: cfg[k] for k in ("T", "v_0", "k", "rho", "theta", "sigma") if k in cfg}
    with E.Engine(NTPB=cfg["NTPB"], NB=cfg["NB"], N=cfg["N"], method=E.METHOD_EM, rng=rng_e, **kw) as e:
        e.init(seed)
        for call in range(2):
            m = e.compute()
            r = ref[call]
            assert r["cuda"] == "cudaSuccess"
            assert _rel(m.mean, r["E"]) < 1e-5, (call, m.mean, r["E"])
            assert _rel(m.variance, r["E2"] - r["E"] ** 2) < 1e-5, (call, m.variance)


def test_compat_reproduces_reference_bias():
    # SURVEY.md §7-4: the reference EM is biased low (E = 0.11718 at 2^18 paths, -7.5 SE vs analytic)
    n = 1 << 18
    with em_engine(n, 1000, rng=1) as e:
        e.init(1234)
        m = e.compute()
    assert (m.mean - o.heston_call()) / m.std_error < -5
    assert abs(m.mean - 0.117179976) < 2 * m.std_error


# ---------------------------------------------------------------------------------------------
# native mode: statistically exact
# ---------------------------------------------------------------------------------------------
def test_native_matches_analytic_and_martingale():
    n = 1 << 20
    with em_engine(n, 1000, rng=0) as e:
        e.init(1234)
        S, V, m = e.compute_paths()
    assert abs(m.mean - o.heston_call()) < 3 * m.std_error, (m.mean, m.std_error)
    se_S = S.astype(np.float64).std() / np.sqrt(n)
    assert abs(S.astype(np.float64).mean() - 1.0) < 3.5 * se_S
    # E[V_T] = theta + (v0 - theta) e^{-kT} = 0.1 at the README point
    assert abs(V.astype(np.float64).mean() - 0.1) < 3.5 * V.astype(np.float64).std() / np.sqrt(n)
    # the oracle's exact-sampler restatement of the same scheme
    ref = o.em_exact_run(o.Params(), seed=3, n_paths=1 << 16)
    se = np.hypot(m.std_error, o.std_error(ref["mean"], ref["mean_sq"], 1 << 16))
    assert abs(m.mean - ref["mean"]) < 3 * se


@pytest.mark.parametrize("k,theta,sigma", [
    (0.5, 0.1, 0.3),             # split, boost recycled from the accept test (the README point)
    (0.5, 0.1, 0.42),            # split, boosted gamma of shape 0.067
    (2.08, 0.108, 0.28),         # split without boost
    (2.08, 0.108, 1.0),          # Poisson mixture: PTRS + inversion + per-lane gamma shape
    (0.1, 0.5, 1.0),             # Poisson mixture, d = 0.1
])
def test_native_tracks_the_oracle_restatement_per_path(k, theta, sigma):
    """The native sampler against the oracle's restatement of ITS mapping (same Philox words, bit fields, trial order,
    recycled boost, commit logic, block counter shared by aligned groups of 32 paths; libm instead of MUFU).  A flipped
    accept/reject re-routes a path, so: the overwhelming majority of paths to 2e-3, the aggregate to a fraction of an SE.
    Two consecutive calls (two streams), a ragged path count, and a shard that starts at path 4096."""
    n, N = 4096 + 37, 60
    p = o.Params(N=N, k=k, theta=theta, sigma=sigma)
    with em_engine_n(n, N, k=k, theta=theta, sigma=sigma) as e:
        e.init(4321)
        for call in range(2):
            S, V, m = e.compute_paths()
            ref = o.em_native_run(p, seed=4321, n_paths=n, call=call, want_paths=True)
            close = np.isclose(S, ref["S"], rtol=2e-3, atol=2e-4) & np.isclose(V, ref["V"], rtol=2e-3, atol=1e-5)
            assert close.mean() > 0.98, (call, close.mean())
            se = o.std_error(ref["mean"], ref["mean_sq"], n)
            assert abs(m.mean - ref["mean"]) < 0.5 * se, (call, m.mean, ref["mean"], se)
    with E.Engine(NTPB=1, NB=1, N=N, method=E.METHOD_EM, n_paths=3 * 4096, first_path=4096, n_local=1000, k=k, theta=theta,
                  sigma=sigma) as e:
        e.init(4321)
        S, V, m = e.compute_paths()
    ref = o.em_native_run(p, seed=4321, first_path=4096, n_paths=1000, want_paths=True)
    assert np.isclose(S, ref["S"], rtol=2e-3, atol=2e-4).mean() > 0.98


@pytest.mark.parametrize("k,theta,sigma,v0", [
    (0.5, 0.1, 0.3, 0.1),        # d = 1.11: split with the boosted gamma (shape 0.61), the boost recycled from the accept test
    (0.5, 0.1, 0.42, 0.1),       # d = 0.567: boosted gamma of shape 0.067
    (0.5, 0.1, 0.32, 0.002),     # d = 0.98 and a small noncentrality: the gamma term dominates
    (10.0, 0.5, 1.0, 0.1),       # d = 10: split without boost
    (2.08, 0.108, 0.28, 0.1),    # d = 5.7
    (2.08, 0.108, 1.0, 0.1),     # d = 0.449: Poisson mixture
    (0.1, 0.5, 1.0, 0.05),       # d = 0.1: Poisson mixture, boosted gamma when N = 0
])
def test_native_one_step_is_the_exact_cir_transition(k, theta, sigma, v0):
    """One step of the native sampler against the exact law of the CIR transition,
    V' = (c / 2) * noncentral-chi-square(df = 2 d, nc = 2 lc V_0)  (NMCH_EM.cu:226-241 in distribution).
    Kolmogorov-Smirnov on 2^18 paths, two consecutive calls (two streams)."""
    from scipy import stats
    n, dt = 1 << 18, 1e-3
    e_kdt = np.exp(-k * dt)
    c = sigma * sigma * (1.0 - e_kdt) / (2.0 * k)
    d = 2.0 * k * theta / (sigma * sigma)
    lc = 2.0 * k * e_kdt / (sigma * sigma * (1.0 - e_kdt))
    law = stats.ncx2(df=2.0 * d, nc=2.0 * lc * v0, scale=0.5 * c)
    with em_engine(n, 1, rng=0, k=k, theta=theta, sigma=sigma, v_0=v0, T=dt) as e:
        e.init(2024)
        for _ in range(2):
            _, V, _ = e.compute_paths()
            V = V.astype(np.float64)
            assert np.isfinite(V).all() and (V >= 0).all()
            ks = stats.kstest(V, law.cdf)
            assert ks.pvalue > 1e-3, (ks, V.mean(), law.mean())
            assert abs(V.mean() - law.mean()) < 4.5 * law.std() / np.sqrt(n)


@pytest.mark.parametrize("k,theta,sigma,want", [
    (2.08, 0.108, 1.0, 0.1104934558),     # d = 0.449 < 1/2: Poisson-mixture path (PTRS + inversion)
    (10.0, 0.5, 1.0, 0.2607554745),       # d = 10: chi-square split, no boost
    (0.1, 0.5, 1.0, 0.0984643143),        # d = 0.1: strongly Feller-violating
    (2.08, 0.108, 0.28, 0.1255567186),    # d = 5.7
    (0.5, 0.1, 0.42, None),               # d = 0.567: split with a boosted gamma of shape 0.067
])
def test_native_parameter_regimes(k, theta, sigma, want):
    n = 1 << 19
    with em_engine(n, 200, rng=0, k=k, theta=theta, sigma=sigma) as e:
        e.init(99)
        S, V, m = e.compute_paths()
    want = want if want is not None else o.heston_call(kappa=k, theta=theta, sigma=sigma)
    # the scheme's only bias is the trapezoid integral of V (O(dt^2)); allow 1e-4 on top of 3.5 SE
    assert abs(m.mean - want) < 3.5 * m.std_error + 1e-4, (m.mean, want, m.std_error)
    S64 = S.astype(np.float64)
    assert abs(S64.mean() - 1.0) < 4 * S64.std() / np.sqrt(n) + 1e-4
    ev = theta + (0.1 - theta) * np.exp(-k)
    V64 = V.astype(np.float64)
    assert abs(V64.mean() - ev) < 4 * V64.std() / np.sqrt(n) + 1e-5


def test_native_general_r_S0_T():
    n = 1 << 19
    with em_engine(n, 200, rng=0, r=0.03, S_0=2.0, T=0.5) as e:
        e.init(7)
        S, V, m = e.compute_paths()
    want_fwd = 2.0 * np.exp(0.03 * 0.5)
    S64 = S.astype(np.float64)
    assert abs(S64.mean() - want_fwd) < 4 * S64.std() / np.sqrt(n)
    # undiscounted payoff mean vs analytic (the reference reports the undiscounted E[(S_T-K)^+])
    want = o.heston_call(S0=2.0, K=2.0, r=0.03, T=0.5) * np.exp(0.03 * 0.5)
    assert abs(m.mean - want) < 3.5 * m.std_error + 2e-4


def test_native_deterministic_sharded_and_streams_advance():
    n, N = 1 << 15, 100
    with em_engine(n, N) as e:
        e.init(5)
        a = e.compute()
        b = e.compute()
    with em_engine(n, N) as e:
        e.init(5)
        a2 = e.compute()
    assert a.sum_payoff == a2.sum_payoff and a.sum_payoff != b.sum_payoff
    parts = []
    for g in range(2):
        with E.Engine(NTPB=512, NB=n // 512, N=N, method=E.METHOD_EM, first_path=g * n // 2, n_local=n // 2) as e:
            e.init(5)
            parts.append(e.compute())
    assert abs(parts[0].sum_payoff + parts[1].sum_payoff - a.sum_payoff) < 1e-9 * n


@pytest.mark.parametrize("rng", [0, 1, 2, 3])
def test_explore_equals_sequential_computes(rng):
    k, th, sg = o.exploration_grid(5, apply_filter=True)
    sel = [0, 7, 40, 120, 199]
    k, th, sg = k[sel], th[sel], sg[sel]
    with em_engine(5120, 50, rng=rng) as e:
        e.init(1234)
        batched = e.explore(k, th, sg)
    with em_engine(5120, 50, rng=rng) as e:
        e.init(1234)
        seq = []
        for i in range(len(k)):
            e.set_params(float(k[i]), float(th[i]), float(sg[i]))
            seq.append(e.compute())
    for b, s in zip(batched, seq):
        assert b.sum_payoff == s.sum_payoff and b.sum_payoff_sq == s.sum_payoff_sq


def test_full_size_properties_2_pow_22():
    # BASELINE configs[2] size (EM, N = 1000, 2^22 paths): size-independent checks
    n = 1 << 22
    with em_engine(n, 1000) as e:
        e.init(1234)
        a = e.compute()
    with em_engine(n, 1000) as e:
        e.init(1234)
        b = e.compute()
    assert a.sum_payoff == b.sum_payoff and a.sum_payoff_sq == b.sum_payoff_sq          # deterministic
    halves = []
    for g in range(2):
        with E.Engine(NTPB=512, NB=n // 512, N=1000, method=E.METHOD_EM, first_path=g * n // 2, n_local=n // 2) as e:
            e.init(1234)
            halves.append(e.compute())
    assert abs(halves[0].sum_payoff + halves[1].sum_payoff - a.sum_payoff) < 1e-10 * n   # shards add up
    assert abs(a.mean - o.heston_call()) < 3 * a.std_error                               # unbiased at 8.6e-5


def test_degenerate_parameters_are_rejected_not_hung():
    from nmch_b200 import capi
    for kw in (dict(sigma=0.0), dict(k=0.0), dict(k=-1.0), dict(theta=float("nan")), dict(v_0=-0.1)):
        for method in (E.METHOD_EM, E.METHOD_QE):
            with E.Engine(NTPB=32, NB=4, N=10, method=method, **kw) as e:
                e.init(1)
                with pytest.raises(capi.NmchError) as ei:
                    e.compute()
                assert ei.value.status == capi.ERR_ARG
    with em_engine(128, 10) as e:                     # setters are validated at the next compute, like the reference's
        e.init(1)
        e.set_params(0.5, 0.1, 0.0)
        with pytest.raises(capi.NmchError):
            e.compute()
        e.set_params(0.5, 0.1, 0.3)
        assert e.compute().n_paths == 128
