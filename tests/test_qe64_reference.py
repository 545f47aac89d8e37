"""Pins the float64 QE-M reference (tests/qe64_reference.py) without the kernel's derivation, CPU only.

Its variance step against the first two moments of the CIR transition, and its log-price step against the martingale
condition, both by quadrature over the step's own draws; its paths against the oracle's float32 restatement of the
kernel on the same Philox words; its absorbed limit at theta = 0; its price against the semi-analytic Heston price."""
import numpy as np
import pytest

import qe64_reference as R
from oracle import oracle as o

README = dict(k=0.5, rho=-0.7, theta=0.1, sigma=0.3)
MODELS = [README, dict(k=2.08, rho=-0.7, theta=0.108, sigma=1.0), dict(k=10.0, rho=-0.7, theta=0.5, sigma=1.0),
          dict(k=1.5, rho=0.9, theta=0.09, sigma=0.5), dict(k=0.5, rho=-0.7, theta=0.1, sigma=1e-3),
          dict(k=1.0, rho=0.5, theta=0.02, sigma=1.0)]
V_GRID = np.array([0.0, 1e-4, 1e-3, 0.01, 0.05, 0.1, 0.3, 1.0, 2.0])


def _hermite(n=80):
    """Nodes and weights of E[f(Z)], Z ~ N(0, 1)."""
    z, w = np.polynomial.hermite_e.hermegauss(n)
    return z, w / np.sqrt(2.0 * np.pi)


def _quadratic_expectation(c, V, f):
    """E[f(V', ln M, Z_v)] over Z_v at a level V of the psi <= 1.5 branch."""
    z, w = _hermite()
    Vn, lnM, psi, quad, _, _ = R.step(c, np.full_like(z, V), z, np.full_like(z, 0.5))
    assert quad.all(), (V, psi)
    return float(np.sum(w * f(Vn, lnM)))


def _exponential_expectation(c, V, f, gamma=1.0):
    """E[f(V', ln M)] over U at a level V of the psi > 1.5 branch: the point mass U <= p (evaluated at U = p / 2), and
    U = 1 - (1 - p) e^{-t} for the tail, where V' = t / beta, by Gauss-Laguerre in tau = gamma t (gamma > 0 scales the
    nodes to an integrand that decays like e^{-gamma t}).  Nodes where U rounds to 1 carry weight below 1e-15 and are
    left out."""
    m, s2 = R.moments(c, V)
    p, _ = R.exponential(s2 / (m * m), m)
    tau, w = np.polynomial.laguerre.laggauss(24)
    t = tau / gamma
    u = np.concatenate([[0.5 * p], 1.0 - (1.0 - p) * np.exp(-t)])
    wt = np.concatenate([[p], (1.0 - p) * w * np.exp(tau - t) / gamma])
    keep = u < 1.0
    assert wt[~keep].sum() < 1e-15
    Vn, lnM, psi, quad, _, _ = R.step(c, np.full(keep.sum(), float(V)), np.zeros(keep.sum()), u[keep])
    assert not quad.any(), (V, psi)
    return float(np.sum(wt[keep] * f(Vn, lnM)))


def _levels(c, branch):
    m, s2 = R.moments(c, V_GRID)
    with np.errstate(divide="ignore", invalid="ignore"):
        psi = s2 / (m * m)
    return [float(v) for v, q in zip(V_GRID, psi) if m[list(V_GRID).index(v)] > 0 and (q <= 1.5) == (branch == "quadratic")]


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("branch", ["quadratic", "exponential"])
def test_variance_step_matches_the_cir_mean_and_variance(model, branch):
    c = R.coefs(1.0, N=50, **model)
    expect = _quadratic_expectation if branch == "quadratic" else _exponential_expectation
    levels = _levels(c, branch)
    for V in levels:
        m, s2 = R.moments(c, V)
        mean = expect(c, V, lambda Vn, lnM: Vn)
        var = expect(c, V, lambda Vn, lnM: (Vn - m) ** 2)
        assert abs(mean / m - 1.0) < 1e-10, (V, mean, m)
        assert abs(var / s2 - 1.0) < 1e-8, (V, var, s2)


def test_both_branches_are_exercised_by_the_moment_checks():
    """Every model has levels on the quadratic side; two (one with rho > 0) reach the exponential side."""
    cs = [R.coefs(1.0, N=50, **model) for model in MODELS]
    assert all(_levels(c, "quadratic") for c in cs)
    assert [len(_levels(c, "exponential")) > 2 for c in cs] == [False, True, False, False, False, True]


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("r", [0.0, 0.05])
def test_log_price_step_is_a_martingale(model, r):
    """E[exp(ln S' - ln S) | V] = e^{r dt} wherever the correction M exists: the check of ln M and of K0*."""
    c = R.coefs(1.0, N=50, **model)
    zs, ws = _hermite()
    # the Z_s integral, by quadrature, of exp(increment) for each (V', ln M)
    def g(V):
        return lambda Vn, lnM: np.array([np.sum(ws * np.exp(R.log_increment(c, r, V, v, l, zs))) for v, l in zip(Vn, lnM)])
    checked = 0
    for V in _levels(c, "quadratic"):
        m, s2 = R.moments(c, V)
        a, _ = R.quadratic(s2 / (m * m), m)
        if 1.0 - 2.0 * c.A * a <= 0.1:
            continue
        got = _quadratic_expectation(c, V, g(V))
        assert abs(got / np.exp(r * c.dt) - 1.0) < 1e-11, (V, got)
        checked += 1
    for V in _levels(c, "exponential"):
        m, s2 = R.moments(c, V)
        p, beta = R.exponential(s2 / (m * m), m)
        if beta <= c.A:
            continue
        got = _exponential_expectation(c, V, g(V), gamma=1.0 - c.A / beta)
        assert abs(got / np.exp(r * c.dt) - 1.0) < 1e-11, (V, got)
        checked += 1
    assert checked >= 5


def test_martingale_correction_exists_in_the_fuzz_box_with_positive_rho():
    """1 - 2 A a > 0 and beta > A for V in [0, 2] over random configurations of test_gpu_fuzz's box with rho in
    [0.2, 0.9]: the correction never has to be clamped there."""
    r = np.random.default_rng(11)
    V = np.linspace(0.0, 2.0, 401)
    for _ in range(400):
        c = R.coefs(float(r.choice([0.25, 0.5, 1.0, 2.0])), k=float(r.uniform(0.2, 6.0)), rho=float(r.uniform(0.2, 0.9)),
                    theta=float(r.uniform(0.02, 0.4)), sigma=float(r.uniform(0.1, 0.9)), N=int(r.integers(1, 120)))
        _, _, _, _, _, exists = R.step(c, V, np.zeros_like(V), np.full_like(V, 0.5))
        assert exists.all(), c


ORACLE_CASES = [
    (dict(), 0, 40),
    (dict(k=2.08, theta=0.108, sigma=1.0), 0, 40),
    (dict(k=10.0, theta=0.5, sigma=1.0), 4096, 40),
    (dict(T=0.5, S_0=100.0, v_0=0.04, r=0.03, k=1.5, rho=-0.3, theta=0.09, sigma=0.5), (1 << 32) - 1000, 17),
    (dict(rho=0.9), 1 << 32, 40),
    (dict(sigma=1e-3), 0, 40),
    (dict(sigma=0.01), 0, 1),
    (dict(theta=0.0), 0, 40),
    (dict(theta=0.0, v_0=0.0, r=0.05), 0, 10),
    (dict(theta=1e-20, S_0=0.5), 0, 40),
]
# Per path, float32 (the oracle, libm) against float64 on identical words, over ORACLE_CASES: S_T to 2.6e-6 (theta = 0),
# 5.7e-7 at sigma = 1e-3 and 1.2e-6 at the README point; V_T to 3.5e-4 relative to |V| + 1e-2 mean V.  Before the
# log-price step was written without cancellation, S_T differed by 2.8e-4 at sigma = 1e-3.
RTOL_S = 2.5e-5
RTOL_V = 3.5e-3
PSI_MARGIN, U_MARGIN = 1e-3, 1e-5


@pytest.mark.parametrize("kw,first,N", ORACLE_CASES)
def test_paths_match_the_oracle_float32_restatement(kw, first, N):
    n, seed, call = 2048, 0xC0FFEE0012345678, 3
    ref = R.qe_paths(**kw, N=N, seed=seed, first_path=first, n_paths=n, call=call)
    orc = o.qe_run(o.Params(N=N, **kw), seed=seed, first_path=first, n_paths=n, call=call, want_paths=True)
    ok = (ref.psi_margin > PSI_MARGIN) & (ref.u_margin > U_MARGIN)
    assert ok.mean() > 0.97 and not ref.no_martingale.any(), (ok.mean(), kw)
    np.testing.assert_allclose(orc["S"][ok], ref.S[ok], rtol=RTOL_S)
    vs = ref.V.mean()
    assert np.all(np.abs(orc["V"][ok] - ref.V[ok]) <= RTOL_V * (ref.V[ok] + 1e-2 * vs)), kw


def test_absorbed_at_zero_when_theta_is_zero():
    """theta = 0: a step from V = 0 stays at 0 for every draw and grows ln S by exactly r dt; from v_0 = 0 every path
    ends at S_0 e^{rT}, and from v_0 > 0 some paths reach 0."""
    c = R.coefs(1.0, k=0.5, rho=-0.7, theta=0.0, sigma=0.3, N=20)
    z = np.linspace(-5.0, 5.0, 101)
    u = np.linspace(0.0, 1.0, 101, endpoint=False) + 0.005
    Vn, lnM, _, _, _, exists = R.step(c, np.zeros_like(z), z, u)
    assert (Vn == 0.0).all() and (lnM == 0.0).all() and exists.all()
    assert np.array_equal(R.log_increment(c, 0.05, 0.0, Vn, lnM, z), np.full_like(z, 0.05 * c.dt))
    p = R.qe_paths(S_0=2.0, v_0=0.0, r=0.05, theta=0.0, N=20, n_paths=512)
    assert (p.V == 0.0).all()
    np.testing.assert_allclose(p.S, 2.0 * np.exp(float(np.float32(0.05))), rtol=1e-14)
    q = R.qe_paths(theta=0.0, N=40, n_paths=2048)
    assert np.isfinite(q.S).all() and 0.05 < (q.V == 0.0).mean() < 0.95


@pytest.mark.parametrize("N,bias", [(10, 6e-4), (50, 2e-4)])
def test_price_matches_semi_analytic(N, bias):
    """The discretisation bias stated as in test_gpu_qe: 6e-4 at dt = 0.1, 2e-4 at dt = 0.02 (README point)."""
    n = 1 << 18
    ref = R.qe_paths(N=N, seed=5, n_paths=n)
    pay = np.maximum(ref.S - 1.0, 0.0)
    want = o.heston_call()
    assert abs(pay.mean() - want) < 3.5 * pay.std() / np.sqrt(n) + bias, (pay.mean(), want)
    assert abs(ref.S.mean() - 1.0) < 4 * ref.S.std() / np.sqrt(n)          # E[S_T] = S_0: the martingale correction
