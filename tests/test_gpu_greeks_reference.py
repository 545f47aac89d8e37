"""compute_greeks() and compute_strikes() against the float64 reference of the native FE step and its v_0 tangent
(tests/fe64_reference.py), at the edges the path kernels are tested at: general parameters, N = 1 and odd N, both
floors, 64-bit seeds, ragged shards, first_path beyond 2^32 and shards across it, and passes that start at a seek()
position (placed after a compute() or an explore() in some configurations) on the Philox low-word carry, with and
without a half-block start.  Also: the strike pass for every (method, rng) pair the engine accepts, the stream forms,
and NaN paths."""
import ctypes as C

import numpy as np
import pytest

import fe64_reference as R

pytestmark = pytest.mark.gpu

SEEKS = (0, 2, 6, (1 << 34) - 12, (1 << 34) - 10, (1 << 40) + 2)
STRIKES = np.array([0.7, 0.9, 1.0, 1.05, 1.3], np.float32)
TILE = 512                      # paths per block of fe_tangent_kernel (kTangentPaths x kTangentThreads)

# Tolerances, each at most 10x the largest value measured over CONFIGS (NVIDIA B200, 1000 W power limit).
DELTA_S = 5e-5          # per-path relative error of S_T; measured 3.1e-5 over all paths (the N = 1 configuration
                        # 7, where one step can bring S_T near 0), 9.9e-7 over the isolated top-64 paths
RTOL_S_SUMS = 2.5e-5    # payoff, payoff^2, delta and itm sums outside the reference bounds, relative to the sum of
                        # |terms|; measured 5.4e-7 at K = 0, 2.9e-6 at the quantile strikes
RTOL_B_SUMS = 1.4e-4    # vega and vega^2 sums, likewise; measured 1.4e-5 at K = 0, 1.5e-5 at the quantile strikes
                        # (configuration 3, 2.4x beyond Feller)
RTOL_B_PATH = 2e-4      # per-path dS_T/dv_0, relative to |B| + 1e-2 mean |B|; measured 2.3e-5
# Not a tolerance: paths whose pre-floor V' came within KINK (relative to the noise term) of 0 are left out of the
# per-path dS_T/dv_0 comparison.  float32 and float64 may take different sides of the floor's kink there, and the
# tangent jumps; oracle.fe_tangent_run (float32 paths) and the float64 reference differ by up to 0.4 relative at a
# margin of 1e-3 and by less than 1e-3 beyond 1e-2 (CPU, the (2.08, 0.108, 1.0) point).
KINK = 1e-2


def _configs(seed, count):
    """Seeded random configurations in the style of test_gpu_fuzz._configs; the greeks pass of configuration i starts at
    SEEKS[i % 6], so every position of SEEKS is compared with the reference twice."""
    r = np.random.default_rng(seed)
    for i in range(count):
        k, theta = float(r.uniform(0.2, 6.0)), float(r.uniform(0.02, 0.4))
        # at most 4x beyond Feller (sigma^2 = 8 k theta; the (2.08, 0.108, 1.0) point is 2.2x): with |.| and a stronger
        # violation paths reflect off V ~ 0 so often that float32 rounding decorrelates them from any float64 restatement
        sigma = min(float(r.uniform(0.1, 0.9)), float(np.sqrt(8 * k * theta)))
        first = int(r.integers(0, 50)) * 4096
        if i % 4 == 1:
            first += 1 << 32                                 # path_hi = 1
        if i % 4 == 3:
            first = (1 << 32) - 4096                         # the shard straddles path 2^32
        yield dict(T=float(r.choice([0.25, 0.5, 1.0, 2.0])), S_0=float(r.choice([0.5, 1.0, 100.0])),
                   v_0=float(r.uniform(0.01, 0.3)), r=float(r.choice([0.0, 0.01, 0.05])), k=k,
                   rho=float(r.uniform(-0.9, 0.5)), theta=theta, sigma=sigma,
                   N=1 if i in (0, 7) else int(r.integers(1, 60)) * 2 + (i % 2),          # N = 1: no main loop
                   n=int(r.integers(300, 4097)) if i % 4 != 3 else 4096 + 1000,
                   seed=int(r.integers(0, 2 ** 63)) * 2 + int(r.integers(0, 2)), first=first, floor=int(r.integers(0, 2)),
                   seek=SEEKS[i % len(SEEKS)], advance=("none", "compute", "explore")[(i // 2) % 3])


CONFIGS = list(_configs(4242, 12))
PARAMS = ("T", "S_0", "v_0", "r", "k", "rho", "theta", "sigma")


def _engine(c, **over):
    from nmch_b200 import engine as E
    kw = {p: c[p] for p in PARAMS}
    kw.update(over)
    return E.Engine(NTPB=1, NB=1, N=c["N"], floor=c["floor"], n_paths=c["first"] + c["n"], first_path=c["first"],
                    n_local=c["n"], **kw)


def _f32p(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _greek_sums(e, strikes):
    """compute_greeks' raw FP64 sums, shape (n_strikes, 6) in R.SUMS order."""
    from nmch_b200 import capi
    strikes = np.ascontiguousarray(strikes, np.float32)
    out = (capi.NmchGreekMoments * len(strikes))()
    capi.check(e._lib.nmch_engine_compute_greeks(e._h, _f32p(strikes), len(strikes), out))
    return np.array([[m.sum_payoff, m.sum_payoff_sq, m.sum_delta, m.sum_itm, m.sum_vega, m.sum_vega_sq] for m in out])


def _strike_sums(e, strikes):
    """compute_strikes' raw FP64 sums, shape (n_strikes, 4): payoff, payoff^2, delta, itm."""
    from nmch_b200 import capi
    strikes = np.ascontiguousarray(strikes, np.float32)
    out = (capi.NmchStrikeMoments * len(strikes))()
    capi.check(e._lib.nmch_engine_compute_strikes(e._h, _f32p(strikes), len(strikes), out))
    return np.array([[m.sum_payoff, m.sum_payoff_sq, m.sum_delta, m.sum_itm] for m in out])


def _advance(e, c):
    """c["advance"] (nothing, one compute() or a two-point explore()), then seek(c["seek"]): the position the greeks pass
    starts at, whatever the engine ran before."""
    if c["advance"] == "compute":
        e.compute()
    elif c["advance"] == "explore":
        e.explore([c["k"], 1.5 * c["k"]], [c["theta"], c["theta"]], [c["sigma"], 0.5 * c["sigma"]])
    e.seek(c["seek"])
    return c["seek"]


def _outside(x, lo, hi, scale):
    """How far x lies outside [lo, hi], relative to scale (0 inside)."""
    return np.maximum(np.maximum(lo - x, x - hi), 0.0) / np.maximum(scale, 1e-300)


def measure_config(c):
    """Runs one configuration; returns what the assertions of test_greeks_match_the_float64_reference bound."""
    with _engine(c) as e:
        e.init(c["seed"])
        w = _advance(e, c)
        ref = R.fe_paths(**{p: c[p] for p in PARAMS}, N=c["N"], floor=c["floor"], seed=c["seed"], first_path=c["first"],
                         n_paths=c["n"], offset=w)
        strikes = np.concatenate([[0.0], np.quantile(ref.S, [0.05, 0.2, 0.35, 0.5, 0.65, 0.8, 0.95]), [c["S_0"]]])
        agg = _greek_sums(e, strikes)
        # per path without a new API: strikes between consecutive top-64 S_T isolate one path per strike difference
        top = np.argsort(-ref.S, kind="stable")[:64]
        s = ref.S[top]
        mids = np.float32(0.5 * (s[:-1] + s[1:]))
        e.seek(w)
        iso = _greek_sums(e, mids)
        e.seek(w)
        S, V, _ = e.compute_paths()
    out = {"S_path": float(np.max(np.abs(S - ref.S) / np.abs(ref.S)))}
    rel = np.zeros((len(strikes), 6))
    for j, K in enumerate(strikes):
        lo, hi, scale = R.strike_fold_bounds(ref.S, ref.B, K, c["S_0"], DELTA_S)
        rel[j] = _outside(agg[j], lo, hi, scale)
    out["k0_S"], out["k0_B"] = float(rel[0, :4].max()), float(rel[0, 4:].max())
    out["q_S"], out["q_B"] = float(rel[1:, :4].max()), float(rel[1:, 4:].max())
    d = np.diff(np.vstack([np.zeros(6), iso]), axis=0)                  # row i: the path of rank i alone
    gap = s[:-1] - s[1:]
    sep = gap > 4 * DELTA_S * np.abs(s[:-1])                               # strike i separates ranks i and i + 1
    ok = sep & np.concatenate([[True], sep[:-1]])                          # both strikes around rank i separate
    idx = top[:63]
    out["iso_itm"] = bool(np.all(d[ok, 3] == 1.0))
    out["iso_S"] = float(np.max(np.abs(d[ok, 2] * np.float32(c["S_0"]) - ref.S[idx[ok]]) / np.abs(ref.S[idx[ok]]), initial=0))
    bscale = np.abs(ref.B).mean()
    okb = ok & (ref.margin[idx] > KINK)
    out["iso_B"] = float(np.max(np.abs(d[okb, 4] - ref.B[idx[okb]]) / (np.abs(ref.B[idx[okb]]) + 1e-2 * bscale), initial=0))
    out["iso_n"] = int(okb.sum())
    out["iso_lanes"] = sorted({int(i % TILE >= TILE // 2) for i in idx[okb]})
    out["kink_share"] = float((ref.margin <= KINK).mean())
    return out


@pytest.mark.parametrize("i", range(len(CONFIGS)))
def test_greeks_match_the_float64_reference(i):
    c = CONFIGS[i]
    m = measure_config(c)
    assert m["S_path"] < DELTA_S, (m, c)
    # K = 0: every path in the money, the sums are sum S, sum S^2, sum S / S_0, n, sum B, sum B^2
    assert m["k0_S"] < RTOL_S_SUMS and m["k0_B"] < RTOL_B_SUMS, (m, c)
    assert m["q_S"] < RTOL_S_SUMS and m["q_B"] < RTOL_B_SUMS, (m, c)
    assert m["iso_itm"], (m, c)
    assert m["iso_n"] >= 20, (m, c)
    assert m["iso_S"] < DELTA_S and m["iso_B"] < RTOL_B_PATH, (m, c)


def test_isolated_paths_cover_both_paths_of_a_thread():
    """The per-path comparison reaches j = 0 and j = 1 of kTangentPaths (this checks the test, not the kernel)."""
    lanes = set()
    for c in CONFIGS[:4]:
        lanes |= set(measure_config(c)["iso_lanes"])
    assert lanes == {0, 1}


EXACT_CASES = [dict(seek=p) for p in SEEKS] + [dict(first=(1 << 32) + 8192), dict(explore=True), dict(S_0=100.0)]


@pytest.mark.parametrize("case", EXACT_CASES, ids=lambda d: "-".join(f"{k}={v}" for k, v in d.items()))
def test_greeks_reproduce_strikes_and_advance_like_compute_bit_for_bit(case):
    from nmch_b200 import engine as E
    n, N = 4096 + 37, 31
    first = case.get("first", 0)
    kw = dict(NTPB=1, NB=1, n_paths=first + n, first_path=first, n_local=n, N=N, S_0=case.get("S_0", 1.0), r=0.01, T=0.75)
    K = STRIKES * np.float32(kw["S_0"])

    def start(e):
        e.init(0x9E3779B97F4A7C15)
        if "seek" in case:
            e.seek(case["seek"])
        if case.get("explore"):
            e.explore([0.5, 2.0, 1.0], [0.1, 0.2, 0.05], [0.3, 0.5, 0.2])

    with E.Engine(**kw) as a, E.Engine(**kw) as b, E.Engine(**kw) as c:
        for e in (a, b, c):
            start(e)
        sa = _strike_sums(a, K)
        gb = _greek_sums(b, K)
        c.compute()
        after_b, after_c = b.compute(), c.compute()
    assert np.array_equal(sa, gb[:, :4]), (sa, gb)
    assert after_b.sum_payoff == after_c.sum_payoff and after_b.sum_payoff_sq == after_c.sum_payoff_sq


ACCEPTED = [(0, rng) for rng in range(6)] + [(1, rng) for rng in range(4)] + [(2, 0)]


def _host_fold(S, K, S0):
    S = S.astype(np.float32)
    pay = np.maximum(S - np.float32(K), 0).astype(np.float64)
    itm = S > np.float32(K)
    return np.array([pay.sum(), (pay * pay).sum(), (S[itm] * np.float32(1.0 / S0)).astype(np.float64).sum(), itm.sum()])


@pytest.mark.parametrize("method,rng", ACCEPTED)
def test_strike_pass_for_every_accepted_method_and_stream(method, rng):
    from nmch_b200 import engine as E
    n, N = 4096 + 37, 41
    # the reference EM scheme assumes T = S_0 = 1 and r = 0
    model = dict(k=1.5, theta=0.08, sigma=0.4, rho=-0.5) if method == 1 else dict(T=0.5, S_0=100.0, r=0.05, v_0=0.06, rho=-0.4)
    kw = dict(NTPB=1, NB=1, n_paths=8192 + n, first_path=8192, n_local=n, N=N, method=method, rng=rng, **model)
    S0 = model.get("S_0", 1.0)
    K = STRIKES * np.float32(S0)
    with E.Engine(**kw) as e:
        e.init(77)
        S, _, m0 = e.compute_paths()
    with E.Engine(**kw) as e:
        e.init(77)
        res = _strike_sums(e, K)
    for j, k in enumerate(K):
        want = _host_fold(S, k, S0)
        assert abs(res[j, 0] - want[0]) < 1e-9 * n * S0, (j, res[j], want)
        assert abs(res[j, 1] - want[1]) < 1e-9 * n * S0 * S0, (j, res[j], want)
        # the host rounds S * float32(1 / S_0) as the kernel does: only the FP64 summation order differs
        assert abs(res[j, 2] - want[2]) < 1e-9 * n and res[j, 3] == want[3], (j, res[j], want)
    assert abs(res[2, 0] - m0.sum_payoff) < 1e-9 * n * S0                   # K = S_0 is the plain compute() result


def test_stream_forms_equal_the_blocking_forms():
    import torch
    from nmch_b200 import engine as E
    kw = dict(NTPB=1, NB=1, n_paths=3000, N=33, T=0.5, r=0.01)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        dev4 = torch.full((2, 4 * len(STRIKES)), float("nan"), dtype=torch.float64, device="cuda")
        dev6 = torch.full((2, 6 * len(STRIKES)), float("nan"), dtype=torch.float64, device="cuda")
    for dev, call, blocking in ((dev4, "compute_strikes_async", _strike_sums), (dev6, "compute_greeks_async", _greek_sums)):
        with E.Engine(**kw) as a, E.Engine(**kw) as b:
            a.init(99)
            b.init(99)
            getattr(a, call)(stream.cuda_stream, STRIKES, dev[0].data_ptr())
            getattr(a, call)(stream.cuda_stream, STRIKES, dev[1].data_ptr())      # continues the stream
            stream.synchronize()
            got = dev.cpu().numpy()
            for row in range(2):
                assert np.array_equal(got[row], blocking(b, STRIKES).ravel()), (call, row)
        assert not np.array_equal(got[0], got[1])


def test_nan_paths_are_carried_into_every_strike_sum():
    """DESIGN.md row A3: a NaN path makes the sums NaN instead of counting as an out-of-the-money path."""
    from nmch_b200 import engine as E
    kw = dict(NTPB=1, NB=1, n_paths=1000, N=20, v_0=float("nan"))
    K = np.array([0.0, 0.5, 1.0, 2.0], np.float32)
    with E.Engine(**kw) as e:
        e.init(3)
        m = e.compute()
        st = _strike_sums(e, K)
        gr = _greek_sums(e, K)
    assert np.isnan(m.sum_payoff) and np.isnan(m.sum_payoff_sq)
    assert np.isnan(st[:, :3]).all() and (st[:, 3] == 0).all(), st
    assert np.isnan(gr[:, [0, 1, 2, 4, 5]]).all() and (gr[:, 3] == 0).all(), gr
