"""Seeded random configurations: every stream mode against the oracle on the same paths (FE per path; EM and QE
per path for the overwhelming majority / statistically), through the C ABI."""
import numpy as np
import pytest

from oracle import oracle as o

pytestmark = pytest.mark.gpu

RNG_PAIRS = {0: o.RNG_PHILOX, 1: o.RNG_XORWOW, 2: o.RNG_PHILOX, 3: o.RNG_MRG32K3A}


def _configs(seed, count):
    r = np.random.default_rng(seed)
    for _ in range(count):
        yield dict(T=float(r.choice([0.25, 0.5, 1.0, 2.0])), S_0=float(r.choice([0.5, 1.0, 100.0])),
                   v_0=float(r.uniform(0.01, 0.3)), r=float(r.choice([0.0, 0.01, 0.05])), k=float(r.uniform(0.2, 6.0)),
                   rho=float(r.uniform(-0.9, 0.5)), theta=float(r.uniform(0.02, 0.4)), sigma=float(r.uniform(0.1, 0.9)),
                   N=int(r.integers(1, 120)), n=int(r.integers(1, 3000)), seed=int(r.integers(0, 2**63)),
                   first=int(r.integers(0, 50)) * 4096, floor=int(r.integers(0, 2)))


@pytest.mark.parametrize("rng", [0, 1, 2, 3])
def test_fe_random_configurations_match_oracle_per_path(rng):
    from nmch_b200 import engine as E
    for c in _configs(1000 + rng, 12):
        kw = {k: c[k] for k in ("T", "S_0", "v_0", "r", "k", "rho", "theta", "sigma")}
        with E.Engine(NTPB=1, NB=1, N=c["N"], rng=rng, floor=c["floor"], n_paths=c["first"] + c["n"], first_path=c["first"],
                      n_local=c["n"], **kw) as e:
            e.init(c["seed"])
            S, V, m = e.compute_paths()
        ref = o.fe_run(o.Params(N=c["N"], **kw), rng=RNG_PAIRS[rng], floor=c["floor"], seed=c["seed"], first_path=c["first"],
                       n_paths=c["n"], want_paths=True)
        tol = 3e-3 if rng == 0 else 3e-4
        np.testing.assert_allclose(S, ref["S"], rtol=tol, atol=tol * c["S_0"] * 0.1, err_msg=str(c))
        np.testing.assert_allclose(V, ref["V"], rtol=10 * tol, atol=tol, err_msg=str(c))
        assert m.n_paths == c["n"]
        pay = np.maximum(S.astype(np.float64) - c["S_0"], 0)
        assert abs(m.sum_payoff - pay.sum()) <= 1e-6 * max(1.0, pay.sum())


@pytest.mark.parametrize("rng", [1, 2, 3])
def test_em_random_configurations_track_oracle(rng):
    from nmch_b200 import engine as E
    for c in _configs(2000 + rng, 6):
        kw = dict(k=c["k"], theta=c["theta"], sigma=c["sigma"], rho=c["rho"], v_0=c["v_0"])   # the reference EM assumes T = S_0 = 1, r = 0
        n = max(c["n"], 256)
        with E.Engine(NTPB=1, NB=1, N=c["N"], method=E.METHOD_EM, rng=rng, n_paths=c["first"] + n, first_path=c["first"],
                      n_local=n, **kw) as e:
            e.init(c["seed"])
            S, V, m = e.compute_paths()
        ref = o.em_run(o.Params(N=c["N"], **kw), rng=RNG_PAIRS[rng], seed=c["seed"], first_path=c["first"], n_paths=n,
                       want_paths=True)
        close = np.isclose(S, ref["S"], rtol=3e-3, atol=3e-4)
        assert close.mean() > 0.95, (close.mean(), c)


def test_qe_random_configurations_match_restatement():
    from nmch_b200 import engine as E
    # every rho of the box, up to 0.5: the martingale correction exists there (1 - 2 A a > 0 and beta > A for V in
    # [0, 2]; test_qe64_reference.test_martingale_correction_exists_in_the_fuzz_box_with_positive_rho)
    for c in _configs(3000, 10):
        kw = {k: c[k] for k in ("T", "S_0", "v_0", "r", "k", "rho", "theta", "sigma")}
        with E.Engine(NTPB=1, NB=1, N=c["N"], method=E.METHOD_QE, n_paths=c["first"] + c["n"], first_path=c["first"],
                      n_local=c["n"], **kw) as e:
            e.init(c["seed"])
            S, V, m = e.compute_paths()
        ref = o.qe_run(o.Params(N=c["N"], **kw), seed=c["seed"], first_path=c["first"], n_paths=c["n"], want_paths=True)
        ok = np.isclose(S, ref["S"], rtol=5e-3, atol=5e-4 * c["S_0"])
        assert ok.mean() > 0.995, (ok.mean(), c)           # a path sitting on the psi = 1.5 switch may take the other branch
