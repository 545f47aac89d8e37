"""GPU parity tests of the FE hot path, through the C ABI (ctypes -> libnmch_b200.so).

Bars (BASELINE.json north_star):
  * XORWOW-/Philox-compat modes vs the oracle: per-path within 2e-4 relative (host libm vs device
    __sincosf/logf differ in the last bits), aggregates within 2e-5 absolute.
  * compat modes vs the reference's own CUDA build (oracle/_ref/nmch_ref_harness, when shipped):
    1e-5 relative on E[X] and on the variance.
  * native Philox mode: within 3 standard errors of the oracle / reference and of the semi-analytic
    Heston price (+ the O(dt) Euler scheme bias the oracle itself shows).
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


def run_engine(n, N=1000, rng=None, floor=0, seed=1234, calls=1, paths=False, **kw):
    ntpb = min(n, 512)
    with E.Engine(NTPB=ntpb, NB=n // ntpb, N=N, rng=rng, floor=floor, **kw) as e:
        e.init(seed)
        for _ in range(calls - 1):
            e.compute()
        if paths:
            return e.compute_paths()
        return e.compute()


# ---------------------------------------------------------------------------------------------
# compat modes vs the oracle
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rng_e,rng_o", [(1, o.RNG_XORWOW), (2, o.RNG_PHILOX), (3, o.RNG_MRG32K3A)])
@pytest.mark.parametrize("floor", [0, 1])
def test_compat_per_path_matches_oracle(rng_e, rng_o, floor):
    n, N = 4096, 200
    S, V, m = run_engine(n, N, rng=rng_e, floor=floor, paths=True)
    ref = o.fe_run(o.Params(N=N), rng=rng_o, floor=floor, n_paths=n, want_paths=True)
    np.testing.assert_allclose(S, ref["S"], rtol=2e-4, atol=2e-5)
    np.testing.assert_allclose(V, ref["V"], rtol=5e-4, atol=2e-5)
    assert abs(m.mean - ref["mean"]) < 2e-5 and abs(m.mean_sq - ref["mean_sq"]) < 2e-5
    assert m.n_paths == n


def test_compat_xorwow_golden_paths():
    # SURVEY.md §8c per-path pins (seed 1234, README parameters, N = 1000)
    S, V, _ = run_engine(512, 1000, rng=1, paths=True)
    np.testing.assert_allclose(S[:3], [1.04778862, 1.15117562, 1.08905244], rtol=2e-4)
    np.testing.assert_allclose(V[:3], [0.0700202361, 0.0975258127, 0.166186899], rtol=5e-4)


def test_compat_xorwow_c1_aggregate():
    m = run_engine(512 * 512, 1000, rng=1)
    assert abs(m.mean - 0.120281939) < 2e-5
    assert abs(m.mean_sq - 0.045731643) < 2e-5


def test_compat_stream_continues_across_calls():
    n, N = 2048, 64
    S, V, m = run_engine(n, N, rng=1, calls=3, paths=True)
    ref = o.fe_run(o.Params(N=N), rng=o.RNG_XORWOW, n_paths=n, calls=3, want_paths=True)
    np.testing.assert_allclose(S, ref["S"], rtol=2e-4, atol=2e-5)
    S, V, m = run_engine(n, 63, rng=2, calls=3, paths=True)          # odd N: Philox resumes mid-block
    ref = o.fe_run(o.Params(N=63), rng=o.RNG_PHILOX, n_paths=n, calls=3, want_paths=True)
    np.testing.assert_allclose(S, ref["S"], rtol=2e-4, atol=2e-5)


def test_compat_shard_offsets_select_subsequences():
    n, N = 8192, 50
    full = o.fe_run(o.Params(N=N), rng=o.RNG_XORWOW, n_paths=n, want_paths=True)
    with E.Engine(NTPB=512, NB=n // 512, N=N, rng=1, first_path=4096 + 17, n_local=1000) as e:
        e.init(1234)
        S, V, m = e.compute_paths()
    np.testing.assert_allclose(S, full["S"][4113:5113], rtol=2e-4, atol=2e-5)


# ---------------------------------------------------------------------------------------------
# compat modes vs the reference's CUDA build
# ---------------------------------------------------------------------------------------------
def _ref_cuda(plus_floor=False, **flags):
    return harness_rows(plus_floor=plus_floor, timeout=600, **flags)


def _rel(a, b):
    return abs(a - b) / abs(b)


@pytest.mark.parametrize("rng_name,rng_e", [("xorwow", 1), ("philox", 2), ("mrg", 3)])
@pytest.mark.parametrize("cfg", [dict(NTPB=512, NB=512, N=1000), dict(NTPB=128, NB=64, N=333),
                                 dict(NTPB=512, NB=512, N=1000, k=2.08, theta=0.108, sigma=1.0)])
def test_compat_matches_reference_cuda_build(rng_name, rng_e, cfg):
    ref = _ref_cuda(method="fe", rng=rng_name, kernel="k3", repeat=2, **cfg)
    kw = {k: cfg[k] for k in ("k", "theta", "sigma") if k in cfg}
    with E.Engine(NTPB=cfg["NTPB"], NB=cfg["NB"], N=cfg["N"], rng=rng_e, **kw) as e:
        e.init(1234)
        for call in range(2):
            m = e.compute()
            r = ref[call]
            assert r["cuda"] == "cudaSuccess"
            var_ref = r["E2"] - r["E"] ** 2
            # tolerance of the north star: 1e-5 relative on price and variance (the reference's own
            # float-atomic accumulation carries ~1e-6 of noise at this size, SURVEY.md §7-3)
            assert _rel(m.mean, r["E"]) < 1e-5, (call, m.mean, r["E"])
            assert _rel(m.variance, var_ref) < 1e-5, (call, m.variance, var_ref)


@pytest.mark.parametrize("seed", [0, 1, 0xFEDCBA9876543210, (1 << 63) + 12345])
@pytest.mark.parametrize("rng_name,modes", [("xorwow", (1, 5)), ("philox", (2, 0)), ("mrg", (3,))])
def test_other_seeds_match_the_reference_cuda_build(seed, rng_name, modes):
    """Seeds beyond 1234: zero, one, and 64-bit seeds whose high half is non-zero (XORWOW scrambles both halves,
    curand_kernel.h:807-818; Philox takes them as its two key words; MRG32k3a derives six state words from them)."""
    cfg = dict(NTPB=256, NB=256, N=200)
    ref = _ref_cuda(method="fe", rng=rng_name, kernel="k3", repeat=2, seed=seed, **cfg)
    for mode in modes:
        with E.Engine(rng=mode, **cfg) as e:
            e.init(seed)
            for call in range(2):
                m = e.compute()
                r = ref[call]
                assert r["cuda"] == "cudaSuccess"
                assert _rel(m.mean, r["E"]) < 1e-5, (mode, seed, call, m.mean, r["E"])
                assert _rel(m.variance, r["E2"] - r["E"] ** 2) < 1e-5, (mode, seed, call)


@pytest.mark.parametrize("rng_name,modes", [("xorwow", (1, 5)), ("philox", (2, 0)), ("mrg", (3,))])
@pytest.mark.parametrize("cfg", [dict(NTPB=512, NB=512, N=1000), dict(NTPB=512, NB=512, N=1000, k=2.08, theta=0.108, sigma=1.0)])
def test_plus_floor_matches_the_reference_cuda_build_with_its_floor_token_changed(rng_name, modes, cfg):
    """BASELINE configs[1] ("|.| floor vs (.)+ floor ... vs reference CUDA build"): the reference codes only abs, so the
    other side is its build with `Vt = abs(Vt);` compiled as `Vt = fmaxf(Vt, 0.0f);` (oracle/Makefile).  Both the
    draw-compatible mode of the tag and the fast mode on the same draws (XORWOW_FAST / native Philox) hold 1e-5."""
    ref = _ref_cuda(plus_floor=True, method="fe", rng=rng_name, kernel="k3", repeat=2, **cfg)
    kw = {k: cfg[k] for k in ("k", "theta", "sigma") if k in cfg}
    for mode in modes:
        with E.Engine(NTPB=cfg["NTPB"], NB=cfg["NB"], N=cfg["N"], rng=mode, floor=E.FLOOR_PLUS, **kw) as e:
            e.init(1234)
            for call in range(2):
                m = e.compute()
                r = ref[call]
                assert r["cuda"] == "cudaSuccess"
                assert _rel(m.mean, r["E"]) < 1e-5, (mode, call, m.mean, r["E"])
                assert _rel(m.variance, r["E2"] - r["E"] ** 2) < 1e-5, (mode, call, m.variance, r["E2"] - r["E"] ** 2)


# ---------------------------------------------------------------------------------------------
# native Philox mode
# ---------------------------------------------------------------------------------------------
def test_native_per_path_tracks_oracle_philox():
    # same Philox words per (path, step) AND (round 2) the same uniforms as cuRAND forms from them; only the
    # transcendentals differ (MUFU lg2 / sqrt against IEEE logf / sqrtf; the sine and cosine are the same MUFU path).
    # Measured on B200 at N = 100: S to 1.4e-6, V to 5.9e-6 (round 1, with bit-spliced 23-bit uniforms: 2e-3 / 1e-2).
    n, N = 4096, 100
    S, V, m = run_engine(n, N, rng=0, paths=True)
    ref = o.fe_run(o.Params(N=N), rng=o.RNG_PHILOX, n_paths=n, want_paths=True)
    np.testing.assert_allclose(S, ref["S"], rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(V, ref["V"], rtol=1e-4, atol=2e-6)


@pytest.mark.parametrize("floor", [0, 1])
def test_native_price_within_3se(floor):
    n = 1 << 20
    m = run_engine(n, 1000, rng=0, floor=floor)
    # vs the semi-analytic Heston price (Euler bias at the README point is below 1e-4, cf. the reference's
    # own 2^24-path XORWOW run: 0.119728 vs 0.119733)
    assert abs(m.mean - o.heston_call()) < 3 * m.std_error + 1e-4
    # vs the reference's arithmetic on the SAME Philox words (compat mode == reference CUDA build to 1e-5):
    # the two estimates are almost perfectly correlated, so they must agree far inside one standard error
    c = run_engine(n, 1000, rng=2, floor=floor)
    assert abs(m.mean - c.mean) < 0.25 * m.std_error, (m.mean, c.mean, m.std_error)
    assert abs(m.variance - c.variance) < 5e-3 * c.variance


def test_native_vs_oracle_same_paths_full_length():
    n = 1 << 13
    S, V, m = run_engine(n, 1000, rng=0, paths=True)
    ref = o.fe_run(o.Params(), rng=o.RNG_PHILOX, n_paths=n, want_paths=True)
    # 1000 steps of ~2^-22 relative transform error per draw on identical uniforms: measured median 9e-7, max 9.8e-6
    np.testing.assert_allclose(S, ref["S"], rtol=1e-4, atol=1e-5)
    assert abs(m.mean - ref["mean"]) < 0.02 * m.std_error


def test_native_feller_violating_point_floors_differ():
    n = 1 << 20
    kw = dict(k=2.08, theta=0.108, sigma=1.0)
    a = run_engine(n, 1000, rng=0, floor=0, **kw)
    p = run_engine(n, 1000, rng=0, floor=1, **kw)
    # SURVEY.md §8c: abs 0.112979, plus 0.111989 (SE 3e-4 at 2^18)
    assert abs(a.mean - 0.112979494) < 4 * 3.0e-4
    assert abs(p.mean - 0.111988764) < 4 * 3.0e-4
    assert a.mean > p.mean


def test_native_paths_per_thread_and_block_size_do_not_change_paths():
    n, N = 8192, 77
    base = run_engine(n, N, rng=0, paths=True, paths_per_thread=1)
    for P, bt in [(2, 256), (4, 256), (8, 256), (4, 128)]:
        S, V, m = run_engine(n, N, rng=0, paths=True, paths_per_thread=P, block_threads=bt)
        np.testing.assert_array_equal(S, base[0])
        np.testing.assert_array_equal(V, base[1])
        assert abs(m.sum_payoff - base[2].sum_payoff) < 1e-9 * n


def test_native_deterministic_and_stream_continues():
    a = run_engine(1 << 16, 100, rng=0)
    b = run_engine(1 << 16, 100, rng=0)
    assert a.sum_payoff == b.sum_payoff and a.sum_payoff_sq == b.sum_payoff_sq
    c = run_engine(1 << 16, 100, rng=0, calls=2)
    assert c.sum_payoff != a.sum_payoff
    # second call of an odd-N run resumes mid-block and equals the oracle's continued stream
    S, V, _ = run_engine(4096, 51, rng=0, calls=2, paths=True)
    ref = o.fe_run(o.Params(N=51), rng=o.RNG_PHILOX, n_paths=4096, calls=2, want_paths=True)
    np.testing.assert_allclose(S, ref["S"], rtol=2e-3, atol=2e-4)


def test_native_sharding_is_additive():
    n, N = 1 << 16, 100
    whole = run_engine(n, N, rng=0)
    parts = []
    for g in range(4):
        with E.Engine(NTPB=512, NB=n // 512, N=N, rng=0, first_path=g * n // 4, n_local=n // 4) as e:
            e.init(1234)
            parts.append(e.compute())
    s = sum(p.sum_payoff for p in parts)
    s2 = sum(p.sum_payoff_sq for p in parts)
    assert abs(s - whole.sum_payoff) < 1e-9 * n and abs(s2 - whole.sum_payoff_sq) < 1e-9 * n


def test_ragged_path_counts():
    for n in (1, 31, 1000, 4097):
        with E.Engine(NTPB=1, NB=n, N=20, rng=0, n_paths=n) as e:
            e.init(5)
            S, V, m = e.compute_paths()
        ref = o.fe_run(o.Params(N=20), rng=o.RNG_PHILOX, seed=5, n_paths=n, want_paths=True)
        np.testing.assert_allclose(S, ref["S"], rtol=2e-3, atol=2e-4)
        assert m.n_paths == n
        assert abs(m.sum_payoff - np.maximum(S.astype(np.float64) - 1.0, 0).sum()) < 1e-6 * max(n, 1)


# ---------------------------------------------------------------------------------------------
# exploration grid in one launch == sequential set_params + compute
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rng", [0, 1, 2, 3])
def test_explore_equals_sequential_computes(rng):
    k, th, sg = o.exploration_grid(5, apply_filter=True)
    k, th, sg = k[:12], th[:12], sg[:12]
    n, N = 5120, 100                                        # the reference's sweep size (exploration.cu:24-25)
    with E.Engine(NTPB=512, NB=10, N=N, rng=rng) as e:
        e.init(1234)
        batched = e.explore(k, th, sg)
    with E.Engine(NTPB=512, NB=10, N=N, rng=rng) as e:
        e.init(1234)
        seq = []
        for i in range(len(k)):
            e.set_params(float(k[i]), float(th[i]), float(sg[i]))
            seq.append(e.compute())
    for b, s in zip(batched, seq):
        assert b.sum_payoff == s.sum_payoff and b.sum_payoff_sq == s.sum_payoff_sq


@pytest.mark.parametrize("rng", [1, 5])
@pytest.mark.parametrize("n,n_points,N", [(5120, 200, 20), (5120 + 77, 37, 33), (1 << 16, 9, 10), (256, 1000, 4)])
def test_xorwow_sweep_in_chunks_equals_the_in_thread_walk(rng, n, n_points, N):
    """XORWOW sweeps (compat and fast) cut the point walk into chunks of consecutive points when the paths cannot fill
    the GPU (the reference's own exploration is 5120 paths x 200 points, exploration.cu:24-25); chunk c starts
    c * chunk_points * 2N draws down each path's stream through the offset skip-ahead.  Same draws per (path, point),
    same blocks per point: the sums are BIT-identical to sequential compute() calls, and the streams continue
    from the same place afterwards."""
    rs = np.random.default_rng(n_points)
    k = rs.uniform(0.1, 5.0, n_points).astype(np.float32)
    th = rs.uniform(0.01, 0.5, n_points).astype(np.float32)
    sg = rs.uniform(0.1, 1.0, n_points).astype(np.float32)
    with E.Engine(NTPB=1, NB=1, N=N, rng=rng, n_paths=n) as e:
        e.init(77)
        batched = e.explore(k, th, sg)
        info = e.launch_info()
        after = e.compute()                                # continues after the sweep
    assert info["grid_y"] > 1 or n >= 148 * 1536, info   # the chunked path is the one under test
    with E.Engine(NTPB=1, NB=1, N=N, rng=rng, n_paths=n) as e:
        e.init(77)
        seq = []
        for i in range(n_points):
            e.set_params(float(k[i]), float(th[i]), float(sg[i]))
            seq.append(e.compute())
        e.set_params(0.5, 0.1, 0.3)
        after_seq = e.compute()
    for i, (b, s_) in enumerate(zip(batched, seq)):
        assert b.sum_payoff == s_.sum_payoff and b.sum_payoff_sq == s_.sum_payoff_sq, i
    assert after.sum_payoff == after_seq.sum_payoff and after.sum_payoff_sq == after_seq.sum_payoff_sq


def test_explore_compat_matches_oracle_sweep():
    k, th, sg = o.exploration_grid(5, apply_filter=True)
    k, th, sg = k[:6], th[:6], sg[:6]
    n, N = 1024, 50
    with E.Engine(NTPB=512, NB=2, N=N, rng=1) as e:
        e.init(1234)
        got = e.explore(k, th, sg)
    sums = o.fe_sweep(o.Params(N=N), k, th, sg, rng=o.RNG_XORWOW, n_paths=n)
    for i, m in enumerate(got):
        assert abs(m.sum_payoff - sums[i, 0]) < 2e-5 * n, i
        assert abs(m.sum_payoff_sq - sums[i, 1]) < 2e-5 * n, i


# ---------------------------------------------------------------------------------------------
# lifecycle / error behaviour
# ---------------------------------------------------------------------------------------------
def test_lifecycle_errors():
    from nmch_b200 import capi
    e = E.Engine(NTPB=32, NB=4, N=10)
    with pytest.raises(capi.NmchError) as ei:
        e.compute()
    assert ei.value.status == capi.ERR_STATE
    e.init(1)
    e.compute()
    e.finalize()
    e.finalize()                                            # idempotent (the reference double-frees)
    with pytest.raises(capi.NmchError):
        e.compute()
    e.close()


# ---------------------------------------------------------------------------------------------
# edge cases: 64-bit path indices and seeds, general r / S_0 / T, single step, size-independent checks
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rng_e,rng_o,tol", [(0, o.RNG_PHILOX, 2e-3), (2, o.RNG_PHILOX, 2e-4), (1, o.RNG_XORWOW, 2e-4)])
def test_paths_beyond_2_pow_32_and_64_bit_seed(rng_e, rng_o, tol):
    first = (1 << 33) + 3 * 4096                      # generator subsequence needs the high counter word
    seed = 0xDEADBEEFCAFEF00D
    n, N = 2048, 60
    with E.Engine(NTPB=1, NB=1, N=N, rng=rng_e, n_paths=first + n, first_path=first, n_local=n) as e:
        e.init(seed)
        S, V, m = e.compute_paths()
    ref = o.fe_run(o.Params(N=N), rng=rng_o, seed=seed, first_path=first, n_paths=n, want_paths=True)
    np.testing.assert_allclose(S, ref["S"], rtol=tol, atol=tol / 10)
    assert abs(m.mean - ref["mean"]) < 10 * tol * 0.2


@pytest.mark.parametrize("rng_e,rng_o,tol", [(0, o.RNG_PHILOX, 3e-3), (1, o.RNG_XORWOW, 2e-4)])
def test_general_rate_spot_maturity(rng_e, rng_o, tol):
    kw = dict(T=0.5, S_0=2.0, v_0=0.04, r=0.03, k=1.5, rho=0.3, theta=0.09, sigma=0.5)
    n, N = 4096, 125
    with E.Engine(NTPB=512, NB=n // 512, N=N, rng=rng_e, **kw) as e:
        e.init(42)
        S, V, m = e.compute_paths()
    ref = o.fe_run(o.Params(N=N, **kw), rng=rng_o, seed=42, n_paths=n, want_paths=True)
    np.testing.assert_allclose(S, ref["S"], rtol=tol, atol=tol)
    np.testing.assert_allclose(V, ref["V"], rtol=10 * tol, atol=tol)
    # payoff is (S_T - S_0)^+ : strike = spot (NMCH.cu:7)
    assert abs(m.sum_payoff - np.maximum(S.astype(np.float64) - 2.0, 0).sum()) < 1e-6 * n


@pytest.mark.parametrize("rng", [0, 1, 2])
def test_single_step_and_single_path(rng):
    with E.Engine(NTPB=1, NB=1, N=1, rng=rng) as e:
        e.init(1234)
        S, V, m = e.compute_paths()
    ref = o.fe_run(o.Params(N=1), rng=o.RNG_XORWOW if rng == 1 else o.RNG_PHILOX, n_paths=1, want_paths=True)
    np.testing.assert_allclose(S, ref["S"], rtol=1e-5)
    np.testing.assert_allclose(V, ref["V"], rtol=1e-4)
    if rng == 1:                                       # SURVEY.md §8c pin: path 0 after one step
        np.testing.assert_allclose([S[0], V[0]], [0.420270562, 0.17408967], rtol=1e-5)


def test_full_size_properties_2_pow_24():
    # BASELINE configs[1] size: checks that do not need an oracle run of that size
    n = 1 << 24
    with E.Engine(NTPB=512, NB=n // 512, N=1000, rng=0) as e:
        e.init(1234)
        a = e.compute()
    with E.Engine(NTPB=512, NB=n // 512, N=1000, rng=0) as e:
        e.init(1234)
        b = e.compute()
    assert a.sum_payoff == b.sum_payoff and a.sum_payoff_sq == b.sum_payoff_sq          # deterministic
    halves = []
    for g in range(2):
        with E.Engine(NTPB=512, NB=n // 512, N=1000, rng=0, first_path=g * n // 2, n_local=n // 2) as e:
            e.init(1234)
            halves.append(e.compute())
    assert abs(halves[0].sum_payoff + halves[1].sum_payoff - a.sum_payoff) < 1e-10 * n   # shards add up
    assert abs(halves[0].sum_payoff_sq + halves[1].sum_payoff_sq - a.sum_payoff_sq) < 1e-10 * n
    assert abs(a.mean - o.heston_call()) < 3 * a.std_error + 5e-5                        # price
    assert 0 < a.variance < a.mean_sq


def test_failed_init_cleans_up_and_reports_cause():
    from nmch_b200 import capi
    e = E.Engine(NTPB=1, NB=1, N=10, rng=1, n_paths=1 << 40)       # 26 TB of XORWOW state: cudaMalloc must fail
    with pytest.raises(capi.NmchError) as ei:
        e.init(1)
    assert ei.value.status == capi.ERR_CUDA and "xorwow states" in str(ei.value) and "cudaErrorMemoryAllocation" in str(ei.value)
    with pytest.raises(capi.NmchError):
        e.compute()
    e.finalize()
    e.close()
    with E.Engine(NTPB=32, NB=4, N=10) as ok:                     # the device is still healthy
        ok.init(1)
        assert ok.compute().n_paths == 128


def test_explore_with_several_tiles_per_block_matches_sequential():
    # many points x many path tiles: blocks walk several tiles each (a different reduction tree than a single compute)
    k, th, sg = o.exploration_grid(5, apply_filter=True)
    k, th, sg = k[:3], th[:3], sg[:3]
    n, N = 1 << 19, 40                                            # 512 tiles of 4 x 256 paths: two tiles per block
    with E.Engine(NTPB=512, NB=n // 512, N=N, rng=0) as e:
        e.init(1234)
        batched = e.explore(k, th, sg)
        assert e.launch_info()["grid_x"] == 256 and e.launch_info()["grid_y"] == 3
    with E.Engine(NTPB=512, NB=n // 512, N=N, rng=0) as e:
        e.init(1234)
        for i in range(3):
            e.set_params(float(k[i]), float(th[i]), float(sg[i]))
            s = e.compute()
            np.testing.assert_allclose([batched[i].sum_payoff, batched[i].sum_payoff_sq], [s.sum_payoff, s.sum_payoff_sq],
                                       rtol=1e-12)


@pytest.mark.parametrize("rng,tol", [(0, 2e-3), (2, 2e-4)])
@pytest.mark.parametrize("offset", [6, (1 << 34) - 12, (1 << 34) - 10, (1 << 40) + 2])
def test_seek_and_block_counter_carry(rng, tol, offset):
    # positions the Philox streams by hand; (2^34 - 12) words = 3 blocks before the LOW counter word wraps, so the
    # 16-step run below crosses the carry into the high word (with and without a half-block start)
    n, N = 2048, 16
    with E.Engine(NTPB=512, NB=n // 512, N=N, rng=rng) as e:
        e.init(1234)
        e.seek(offset)
        S, V, m = e.compute_paths()
        S2, _, _ = e.compute_paths()                      # and the stream keeps going from there
    ref = o.fe_run_at(o.Params(N=N), offset, rng=o.RNG_PHILOX, n_paths=n, calls=2, want_paths=True)
    first = o.fe_run_at(o.Params(N=N), offset, rng=o.RNG_PHILOX, n_paths=n, want_paths=True)
    np.testing.assert_allclose(S, first["S"], rtol=tol, atol=tol / 10)
    np.testing.assert_allclose(S2, ref["S"], rtol=tol, atol=tol / 10)


def test_seek_rejected_outside_philox_fe():
    from nmch_b200 import capi
    with E.Engine(NTPB=32, NB=4, N=10, rng=1) as e:
        e.init(1)
        with pytest.raises(capi.NmchError):
            e.seek(4)
    with E.Engine(NTPB=32, NB=4, N=10, rng=0) as e:
        e.init(1)
        with pytest.raises(capi.NmchError):
            e.seek(3)
