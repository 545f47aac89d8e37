"""Pins the five-direction tangent of the float64 reference (tests/fe64_sensitivity_reference.py: dS / dV), CPU only.

Each direction against a central finite difference of the float64 paths in that parameter (the check that shares no
derivation with the product's step), at both floors, the Feller-violating (2.08, 0.108, 1.0) point, r != 0 and
rho in {-0.9, 0, 0.5}; and the (.)+ floor's parked paths, whose kappa and theta tangents restart from 0."""
import numpy as np
import pytest

import fe64_reference as R
import fe64_sensitivity_reference as RS

FELLER_VIOLATING = dict(k=2.08, theta=0.108, sigma=1.0)
KINK = 1e-2                     # as test_gpu_greeks_reference: paths that came this close to V' = 0 are left out
SHIFT = {"v0": "v0_shift", "kappa": "k_shift", "theta": "theta_shift", "sigma": "sigma_shift", "rho": "rho_shift"}
BASE = {"v0": "v_0", "kappa": "k", "theta": "theta", "sigma": "sigma", "rho": "rho"}
DEFAULTS = dict(v_0=0.1, k=0.5, theta=0.1, sigma=0.3, rho=-0.7)

CASES = [
    dict(N=100),
    dict(N=100, **FELLER_VIOLATING),
    dict(N=60, T=0.5, S_0=100.0, v_0=0.2, r=0.05, rho=-0.9, k=4.0, sigma=0.6),
    dict(N=80, r=0.03, rho=0.0),
    dict(N=80, T=2.0, r=0.01, rho=0.5, **FELLER_VIOLATING),
]


@pytest.mark.parametrize("floor", [0, 1])
@pytest.mark.parametrize("kw", CASES, ids=lambda kw: "-".join(f"{k}={v}" for k, v in kw.items()))
@pytest.mark.parametrize("d", range(5), ids=RS.DIRS)
def test_each_direction_equals_a_central_difference_of_the_float64_paths(floor, kw, d):
    name = RS.DIRS[d]
    run = dict(kw, floor=floor, seed=0x5EED, first_path=8192, n_paths=4096, offset=6)
    p = RS.fe_paths(**run)
    base = float(np.float32(kw.get(BASE[name], DEFAULTS[BASE[name]])))
    h = 1e-6 * max(abs(base), 0.1)
    up = RS.fe_paths(**run, **{SHIFT[name]: h})
    dn = RS.fe_paths(**run, **{SHIFT[name]: -h})
    fd_S = (up.S - dn.S) / (2 * h)
    fd_V = (up.V - dn.V) / (2 * h)
    smooth = p.margin > KINK
    assert smooth.mean() > 0.5
    assert np.isfinite(p.dS).all() and np.isfinite(p.dV).all()
    sS = np.abs(p.dS[d]).mean() + 1e-300
    np.testing.assert_allclose(p.dS[d][smooth], fd_S[smooth], rtol=1e-3, atol=1e-5 * sS)
    if name == "rho":
        assert not p.dV[d].any()                                 # V does not depend on rho
    else:
        sV = np.abs(p.dV[d]).mean() + 1e-300
        np.testing.assert_allclose(p.dV[d][smooth], fd_V[smooth], rtol=1e-3, atol=1e-5 * sV)


def test_v0_direction_is_the_v0_tangent():
    """The v_0 row equals fe64_reference's own v_0 tangent (B = dS/dv_0, A = dV/dv_0) on the same paths."""
    p = RS.fe_paths(N=50, floor=1, n_paths=2048, **FELLER_VIOLATING)
    q = R.fe_paths(N=50, floor=1, n_paths=2048, **FELLER_VIOLATING)
    np.testing.assert_array_equal(p.S, q.S)
    np.testing.assert_array_equal(p.margin, q.margin)
    np.testing.assert_allclose(p.dS[0], q.B, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(p.dV[0], q.A, rtol=1e-12, atol=1e-15)


def test_parked_paths_restart_their_kappa_and_theta_tangents():
    """(.)+ parks a path at V = 0 and zeroes its variance tangents in that step; in the next step the drift k theta dt
    lifts it off 0 again, and the tangents of kappa and theta restart at theta dt and kappa dt, not at 0.  v_0 = 0 starts
    every path parked: after one step V = k theta dt exactly (no noise at V = 0)."""
    T, N, k, theta = 1.0, 1, 2.08, 0.108
    dt = float(np.float32(T) / np.float32(N))
    kf, tf = float(np.float32(k)), float(np.float32(theta))
    p = RS.fe_paths(T=T, N=N, v_0=0.0, k=k, theta=theta, sigma=1.0, floor=R.FLOOR_PLUS, n_paths=64)
    np.testing.assert_allclose(p.V, kf * tf * dt, rtol=1e-15)
    np.testing.assert_allclose(p.dV[1], tf * dt, rtol=1e-15)
    np.testing.assert_allclose(p.dV[2], kf * dt, rtol=1e-15)
    assert not p.dV[3].any() and not p.dS.any()
    # ... and over 40 steps they reach S_T: central differences agree (the floor parks some paths on the way)
    run = dict(T=0.4, N=40, v_0=0.0, floor=R.FLOOR_PLUS, n_paths=4096, **FELLER_VIOLATING)
    p = RS.fe_paths(**run)
    assert (p.V == 0).any() or (p.margin < 1).any()
    smooth = p.margin > KINK
    for d, shift in ((1, "k_shift"), (2, "theta_shift")):
        h = 1e-7
        fd = (RS.fe_paths(**run, **{shift: h}).S - RS.fe_paths(**run, **{shift: -h}).S) / (2 * h)
        assert np.abs(p.dS[d]).max() > 0
        np.testing.assert_allclose(p.dS[d][smooth], fd[smooth], rtol=1e-3, atol=1e-5 * np.abs(p.dS[d]).mean())
