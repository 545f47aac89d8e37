"""SURVEY.md §8 f4, second half: the reference's K1 kernels store E[X^2]/n^2 in price_squared
(/root/reference/src/NMCH/methods/NMCH_FE.cu:56-58, NMCH_EM.cu:129-131: they reduce (payoff/n)^2/n).  Behind
set_legacy_k1_moment(true) / `NMCH --legacy-k1` the K1 classes reproduce that value; checked against the reference's
own K1 classes (oracle/_ref/nmch_ref_harness --kernel k1, the unmodified sources) on identical seeds."""
import json
import os
import subprocess

import pytest

from ref_build import harness_rows

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NMCH = os.path.join(ROOT, "bin", "NMCH")


@pytest.fixture(scope="module", autouse=True)
def _built():
    from nmch_b200 import _build
    _build.build_cli(only_if_missing=True)


def _ours(*args):
    r = subprocess.run([NMCH, *map(str, args), "--json"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-300:] + r.stderr[-300:]
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1]), r.stdout


def _ref(**flags):
    return harness_rows(timeout=600, **flags)


@pytest.mark.parametrize("method,N", [("fe", 200), ("em", 100)])
def test_legacy_k1_moment_matches_the_reference_k1_class(method, N):
    ntpb, nb = 256, 64                                   # K1's shared-memory tree needs a power-of-two NTPB
    n = ntpb * nb
    ref = _ref(method=method, rng="xorwow", kernel="k1", NTPB=ntpb, NB=nb, N=N)[0]
    ref_k3 = _ref(method=method, rng="xorwow", kernel="k3", NTPB=ntpb, NB=nb, N=N)[0]
    # the quirk, as the survey states it: K1's price_squared is K3's divided by n^2
    assert abs(ref["E2"] * n * n - ref_k3["E2"]) < 2e-5 * ref_k3["E2"]
    ours, text = _ours("--method", method, "--rng", "xorwow", "--legacy-k1", "--NTPB", ntpb, "--NB", nb, "--N", N)
    assert abs(ours["E"] - ref["E"]) < 1e-5 * ref["E"]
    assert abs(ours["E2"] - ref["E2"]) < 1e-5 * ref["E2"], (ours["E2"], ref["E2"])
    # the same class without the switch stores E[X^2], like the reference's K2 / K3
    plain, _ = _ours("--method", method, "--rng", "xorwow", "--NTPB", ntpb, "--NB", nb, "--N", N)
    assert abs(plain["E2"] - ref_k3["E2"]) < 1e-5 * ref_k3["E2"]
    assert abs(plain["E2"] / ours["E2"] - float(n) ** 2) < 1e-4 * float(n) ** 2


def test_python_mirror_applies_the_quirk_to_k1_classes_only():
    from nmch_b200 import methods as M
    args = (256, 16, 1.0, 1.0, 0.1, 0.0, 0.5, -0.7, 0.1, 0.3, 50)
    vals = {}
    for cls in (M.NMCH_FE_K1_MM, M.NMCH_FE_K3_MM, M.NMCH_FE_K1_PgM, M.NMCH_EM_K1_MM, M.NMCH_EM_K2_MM):
        m = cls(*args, M.XORWOW)
        m.set_legacy_k1_moment(True)
        m.init(1234)
        m.compute()
        vals[cls.__name__] = (m.get_price_squared(), m.last_moments.mean_sq)
        m.finalize()
    n2 = float(256 * 16) ** 2
    for name in ("NMCH_FE_K1_MM", "NMCH_FE_K1_PgM", "NMCH_EM_K1_MM"):
        got, e2 = vals[name]
        assert abs(got * n2 - e2) < 1e-6 * e2, name
    for name in ("NMCH_FE_K3_MM", "NMCH_EM_K2_MM"):
        got, e2 = vals[name]
        assert abs(got - e2) < 1e-6 * e2, name
