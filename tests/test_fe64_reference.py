"""Pins the float64 reference of the native FE step and its v_0 tangent (tests/fe64_reference.py), CPU only.

Its Philox against the oracle's restatement of cuRAND; its paths against the oracle's IEEE float32 FE run on cuRAND's
Philox stream; its tangent against a central finite difference of its own float64 paths (the check that does not
share the derivation of the product or of oracle.fe_tangent_run) and, where the two should agree, against
oracle.fe_tangent_run."""
import numpy as np
import pytest

import fe64_reference as R
from oracle import oracle as o

FELLER_VIOLATING = dict(k=2.08, theta=0.108, sigma=1.0)
GENERAL = dict(T=0.5, S_0=100.0, v_0=0.2, r=0.05, rho=-0.3, N=77)


def test_philox_matches_the_oracle_across_the_low_word_carry_path_hi_and_a_64_bit_key():
    key = (0x89ABCDEF, 0x01234567)
    blocks = [0, 1, 0xFFFFFFFE, 0xFFFFFFFF, 1 << 32, (1 << 32) + 1, (5 << 32) + 0xFFFFFFFF]
    paths = [0, 7, 0xFFFFFFFF, 1 << 32, (3 << 32) + 12345]
    for blk in blocks:
        ctr = (blk & 0xFFFFFFFF, blk >> 32, np.array([p & 0xFFFFFFFF for p in paths]), np.array([p >> 32 for p in paths]))
        got = R.philox4x32_10(ctr, key)
        for i, p in enumerate(paths):
            want = o.philox4x32_10([blk & 0xFFFFFFFF, blk >> 32, p & 0xFFFFFFFF, p >> 32], list(key))
            assert [int(w[i]) for w in got] == want, (blk, p)


@pytest.mark.parametrize("floor", [0, 1])
@pytest.mark.parametrize("kw,first,offset", [
    (dict(N=60), 0, 0),
    (GENERAL, (1 << 32) + 4096, 6),
    (dict(GENERAL, T=2.0, S_0=0.5, r=0.01, rho=0.4, N=31, **FELLER_VIOLATING), 8192, (1 << 34) - 10),
    (dict(T=0.25, v_0=0.03, N=1), 4096, (1 << 40) + 2),
])
def test_paths_match_the_oracle_float32_run_on_the_same_words(floor, kw, first, offset):
    seed = 0xF00DFACE12345678
    n = 1500
    ref = R.fe_paths(**kw, floor=floor, seed=seed, first_path=first, n_paths=n, offset=offset)
    p = {k: v for k, v in kw.items()}
    orc = o.fe_run_at(o.Params(**p), offset, rng=o.RNG_PHILOX, floor=floor, seed=seed, first_path=first, n_paths=n,
                      want_paths=True)
    # float32 IEEE against float64 on identical words, measured over these cases: S to 3.4e-6; V near 0 is compared
    # absolutely, and V uses at most 0.13 of the bound below
    np.testing.assert_allclose(orc["S"], ref.S, rtol=3e-5)
    np.testing.assert_allclose(orc["V"], ref.V, rtol=2e-4, atol=2e-6)


@pytest.mark.parametrize("floor", [0, 1])
@pytest.mark.parametrize("kw", [dict(N=100), dict(N=100, **FELLER_VIOLATING), dict(GENERAL, rho=0.3, k=4.0, sigma=0.6)])
def test_tangent_equals_a_central_difference_of_the_float64_paths(floor, kw):
    n = 4096
    v0 = float(np.float32(kw.get("v_0", 0.1)))
    h = 1e-6 * v0
    run = dict(kw, floor=floor, seed=77, first_path=4096, n_paths=n, offset=2)
    p = R.fe_paths(**run)
    fd = (R.fe_paths(**run, v0_shift=h).S - R.fe_paths(**run, v0_shift=-h).S) / (2 * h)
    # a path whose pre-floor V' passes within 1e-4 (of the noise term) of 0 may cross the kink inside [v0 - h, v0 + h]
    smooth = p.margin > 1e-4
    assert (~smooth).mean() < 0.01
    scale = np.abs(p.B).mean()
    np.testing.assert_allclose(p.B[smooth], fd[smooth], rtol=1e-3, atol=1e-5 * scale)   # measured: 3e-4


@pytest.mark.parametrize("floor", [0, 1])
def test_kink_paths_are_rare_at_the_feller_violating_point(floor):
    p = R.fe_paths(N=250, floor=floor, n_paths=8192, **FELLER_VIOLATING)
    assert (p.margin <= 1e-4).mean() < 0.01


@pytest.mark.parametrize("floor", [0, 1])
@pytest.mark.parametrize("kw", [dict(N=60), dict(N=100, **FELLER_VIOLATING), dict(GENERAL, N=40)])
def test_tangent_agrees_with_the_oracle_tangent(floor, kw):
    n = 4096
    p = R.fe_paths(**kw, floor=floor, seed=5, n_paths=n)
    t = o.fe_tangent_run(o.Params(**kw), floor=floor, seed=5, n_paths=n)
    # the oracle carries B in double on float32 paths: away from the kink they agree to the float32 path error
    smooth = p.margin > 1e-2
    scale = np.abs(p.B).mean()
    np.testing.assert_allclose(t["B"][smooth], p.B[smooth], rtol=1e-2, atol=1e-4 * scale)


def test_strike_fold_bounds():
    S = np.array([0.5, 0.99999, 1.0, 1.00001, 1.5, 2.0])
    B = np.array([0.1, -0.2, 0.3, 0.4, -0.5, 0.6])
    lo, hi, scale = R.strike_fold_bounds(S, B, 1.0, 1.0, 2e-5)
    # 0.99999, 1.0 and 1.00001 are within 2e-5 of K: each may or may not be in the money
    band = 2e-5 * np.array([1.0, 1.0, 1.00001])
    sure_pay = 0.5 + 1.0
    amb_pay = np.abs(S[1:4] - 1.0) + band
    np.testing.assert_allclose(lo, [sure_pay, 0.25 + 1.0, 3.5, 2, -0.5 + 0.6 - 0.2, 0.25 + 0.36])
    np.testing.assert_allclose(hi[0], sure_pay + amb_pay.sum())
    np.testing.assert_allclose(hi[2:], [3.5 + 3.0, 5, 0.1 + 0.3 + 0.4, 0.61 + 0.04 + 0.09 + 0.16])
    assert (scale >= np.maximum(np.abs(lo), np.abs(hi)) - 1e-12).all()
    lo0, hi0, _ = R.strike_fold_bounds(S, B, 0.0, 1.0, 2e-5)
    np.testing.assert_allclose(lo0, hi0)
    np.testing.assert_allclose(lo0, [S.sum(), (S * S).sum(), S.sum(), 6, B.sum(), (B * B).sum()])
