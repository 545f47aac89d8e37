"""Thin object wrapper over the C ABI: one Engine == one nmch_engine_t handle.

This is host plumbing only (argument packing, numpy views); all arithmetic happens in the CUDA
library.  Mirrors the lifecycle of the reference's method objects (init / compute / finalize,
/root/reference/include/NMCH/methods/NMCH.hpp:42-60).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import capi
from .capi import (FLOOR_ABS, FLOOR_PLUS, METHOD_EM, METHOD_FE, METHOD_QE, RNG_MRG32K3A_COMPAT, RNG_PHILOX,  # noqa: F401
                   RNG_PHILOX_COMPAT, RNG_PHILOX_DENSE, RNG_XORWOW_COMPAT, RNG_XORWOW_FAST)


@dataclass
class Moments:
    """Raw FP64 sums of one compute() pass and the statistics the reference derives from them."""
    sum_payoff: float
    sum_payoff_sq: float
    n_paths: int
    exec_ms: float

    @property
    def mean(self) -> float:            # E[X]   (strike_price in the reference's naming)
        return self.sum_payoff / self.n_paths

    @property
    def mean_sq(self) -> float:         # E[X^2] (price_squared)
        return self.sum_payoff_sq / self.n_paths

    @property
    def variance(self) -> float:
        return max(self.mean_sq - self.mean * self.mean, 0.0)

    @property
    def std_error(self) -> float:
        return float(np.sqrt(self.variance / self.n_paths))

    def merged(self, other: "Moments") -> "Moments":
        return Moments(self.sum_payoff + other.sum_payoff, self.sum_payoff_sq + other.sum_payoff_sq,
                       self.n_paths + other.n_paths, max(self.exec_ms, other.exec_ms))


def _strike_rows(out):
    """Per strike: payoff moments, pathwise delta and in-the-money share."""
    return [{"strike": m.strike, "moments": Moments(m.sum_payoff, m.sum_payoff_sq, m.n_paths, m.exec_ms),
             "delta": m.sum_delta / m.n_paths, "itm": m.sum_itm / m.n_paths} for m in out]


def _greek_rows(out):
    """Per strike: payoff moments, pathwise delta, in-the-money share, pathwise vega (d price / d v_0) and its
    standard error."""
    rows = []
    for m in out:
        n = m.n_paths
        vega = m.sum_vega / n
        var = max(m.sum_vega_sq / n - vega * vega, 0.0)
        rows.append({"strike": m.strike, "moments": Moments(m.sum_payoff, m.sum_payoff_sq, n, m.exec_ms),
                     "delta": m.sum_delta / n, "itm": m.sum_itm / n, "vega_v0": vega,
                     "vega_v0_se": (var / max(n - 1, 1)) ** 0.5})
    return rows


def _sensitivity_rows(out):
    """Per strike: the keys of compute_strikes() (payoff moments, delta, in-the-money share) and, for each parameter p of
    capi.SENS_NAMES, the pathwise d E[(S_T - K)^+] / d p as "d_<p>" and its standard error as "d_<p>_se" (computed as
    _greek_rows computes vega_v0 / vega_v0_se)."""
    rows = []
    for m in out:
        n = m.n_paths
        row = {"strike": m.strike, "moments": Moments(m.sum_payoff, m.sum_payoff_sq, n, m.exec_ms),
               "delta": m.sum_delta / n, "itm": m.sum_itm / n}
        for d, name in enumerate(capi.SENS_NAMES):
            mean = m.sum_sens[d] / n
            var = max(m.sum_sens_sq[d] / n - mean * mean, 0.0)
            row[f"d_{name}"] = mean
            row[f"d_{name}_se"] = (var / max(n - 1, 1)) ** 0.5
        rows.append(row)
    return rows


def _strike_call(fn, handle, strikes, struct, rows):
    """One blocking strike-family call of the C ABI (engine or group): fn(handle, strikes, n, out) into an array of
    `struct`, returned as rows(out)."""
    strikes = np.ascontiguousarray(strikes, np.float32)
    out = (struct * len(strikes))()
    capi.check(fn(handle, strikes.ctypes.data_as(C.POINTER(C.c_float)), len(strikes), out))
    return rows(out)


def _strike_call_async(fn, handle, stream_ptr, strikes, d_moments_ptr):
    """The stream form of _strike_call: raw sums land in device memory at d_moments_ptr."""
    strikes = np.ascontiguousarray(strikes, np.float32)
    capi.check(fn(handle, C.c_void_p(stream_ptr), strikes.ctypes.data_as(C.POINTER(C.c_float)), len(strikes),
                  C.c_void_p(d_moments_ptr)))


class Engine:
    def __init__(self, NTPB=512, NB=512, T=1.0, S_0=1.0, v_0=0.1, r=0.0, k=0.5, rho=-0.7, theta=0.1, sigma=0.3,
                 N=1000, method=METHOD_FE, floor=FLOOR_ABS, rng=RNG_PHILOX, device=-1, n_paths=0, first_path=0,
                 n_local=0, paths_per_thread=0, block_threads=0):
        self._lib = capi.load()
        self.params = capi.NmchParams(NTPB, NB, T, S_0, v_0, r, k, rho, theta, sigma, N, method, floor, rng,
                                      device, n_paths, first_path, n_local, paths_per_thread, block_threads)
        self._h = C.c_void_p()
        capi.check(self._lib.nmch_engine_create(C.byref(self.params), C.byref(self._h)))
        self.n_paths = n_paths or NTPB * NB
        self.n_local = n_local or (self.n_paths - first_path)
        self.N = N

    # -- lifecycle ---------------------------------------------------------------------------
    def init(self, seed: int = 1234) -> "Engine":
        capi.check(self._lib.nmch_engine_init(self._h, seed))
        return self

    def set_params(self, k: float, theta: float, sigma: float) -> None:
        capi.check(self._lib.nmch_engine_set_params(self._h, k, theta, sigma))

    def seek(self, words: int) -> None:
        """Position the streams after `words` 32-bit draws per path (FE, Philox modes)."""
        capi.check(self._lib.nmch_engine_seek(self._h, words))

    def compute(self) -> Moments:
        m = capi.NmchMoments()
        capi.check(self._lib.nmch_engine_compute(self._h, C.byref(m)))
        return Moments(m.sum_payoff, m.sum_payoff_sq, m.n_paths, m.exec_ms)

    def compute_async(self, stream_ptr: int, d_moments_ptr: int) -> None:
        """Enqueue one pass on a caller stream; raw sums land in device memory (2 doubles)."""
        capi.check(self._lib.nmch_engine_compute_async(self._h, C.c_void_p(stream_ptr), C.c_void_p(d_moments_ptr)))

    def explore(self, k, theta, sigma):
        k = np.ascontiguousarray(k, np.float32)
        theta = np.ascontiguousarray(theta, np.float32)
        sigma = np.ascontiguousarray(sigma, np.float32)
        n = len(k)
        out = (capi.NmchMoments * n)()
        f32p = C.POINTER(C.c_float)
        capi.check(self._lib.nmch_engine_explore(self._h, k.ctypes.data_as(f32p), theta.ctypes.data_as(f32p),
                                                 sigma.ctypes.data_as(f32p), n, out))
        return [Moments(m.sum_payoff, m.sum_payoff_sq, m.n_paths, m.exec_ms) for m in out]

    def explore_async(self, stream_ptr: int, k, theta, sigma, d_moments_ptr: int) -> None:
        k = np.ascontiguousarray(k, np.float32)
        theta = np.ascontiguousarray(theta, np.float32)
        sigma = np.ascontiguousarray(sigma, np.float32)
        f32p = C.POINTER(C.c_float)
        capi.check(self._lib.nmch_engine_explore_async(self._h, C.c_void_p(stream_ptr), k.ctypes.data_as(f32p),
                                                       theta.ctypes.data_as(f32p), sigma.ctypes.data_as(f32p),
                                                       len(k), C.c_void_p(d_moments_ptr)))

    def compute_paths(self, count: int | None = None):
        """Parity hook: one compute() pass that also returns terminal S, V of local paths [0, count)."""
        count = self.n_local if count is None else count
        S = np.empty(count, np.float32)
        V = np.empty(count, np.float32)
        m = capi.NmchMoments()
        f32p = C.POINTER(C.c_float)
        capi.check(self._lib.nmch_engine_compute_paths(self._h, S.ctypes.data_as(f32p), V.ctypes.data_as(f32p),
                                                       count, C.byref(m)))
        return S, V, Moments(m.sum_payoff, m.sum_payoff_sq, m.n_paths, m.exec_ms)

    def compute_strikes(self, strikes):
        """One compute() pass priced at a vector of strikes, with the pathwise delta (SURVEY.md §8f rank 2)."""
        return _strike_call(self._lib.nmch_engine_compute_strikes, self._h, strikes, capi.NmchStrikeMoments,
                            _strike_rows)

    def compute_strikes_async(self, stream_ptr: int, strikes, d_moments_ptr: int) -> None:
        """Enqueue compute_strikes() on a caller stream; raw sums land in device memory (4 doubles per strike:
        payoff, payoff^2, delta, in-the-money count)."""
        _strike_call_async(self._lib.nmch_engine_compute_strikes_async, self._h, stream_ptr, strikes, d_moments_ptr)

    def compute_greeks(self, strikes):
        """compute_strikes() plus the pathwise vega d E[(S_T - K)^+] / d v_0 (FE, native Philox stream only)."""
        return _strike_call(self._lib.nmch_engine_compute_greeks, self._h, strikes, capi.NmchGreekMoments, _greek_rows)

    def compute_greeks_async(self, stream_ptr: int, strikes, d_moments_ptr: int) -> None:
        """Enqueue compute_greeks() on a caller stream; raw sums land in device memory (6 doubles per strike:
        payoff, payoff^2, delta, in-the-money count, vega, vega^2)."""
        _strike_call_async(self._lib.nmch_engine_compute_greeks_async, self._h, stream_ptr, strikes, d_moments_ptr)

    def compute_sensitivities(self, strikes):
        """compute_strikes() plus the pathwise sensitivities of E[(S_T - K)^+] to v_0, kappa, theta, sigma and rho from
        the same pass (FE, native Philox stream only; |rho| < 1).  Rows carry "d_v0", "d_kappa", "d_theta", "d_sigma",
        "d_rho" and their standard errors "d_<p>_se"."""
        return _strike_call(self._lib.nmch_engine_compute_sensitivities, self._h, strikes, capi.NmchSensitivityMoments,
                            _sensitivity_rows)

    def compute_sensitivities_async(self, stream_ptr: int, strikes, d_moments_ptr: int) -> None:
        """Enqueue compute_sensitivities() on a caller stream; raw sums land in device memory (14 doubles per strike:
        payoff, payoff^2, delta, in-the-money count, then sum and sum of squares for v_0, kappa, theta, sigma, rho)."""
        _strike_call_async(self._lib.nmch_engine_compute_sensitivities_async, self._h, stream_ptr, strikes,
                           d_moments_ptr)

    def check(self) -> None:
        """Synchronise and, in the checked build, sweep the guard bands / surface a failed device assert."""
        capi.check(self._lib.nmch_engine_check(self._h))

    def finalize(self) -> None:
        if self._h:
            capi.check(self._lib.nmch_engine_finalize(self._h))

    def close(self) -> None:
        if self._h:
            self._lib.nmch_engine_destroy(self._h)
            self._h = C.c_void_p()

    # -- reports -----------------------------------------------------------------------------
    @property
    def init_ms(self) -> float:
        return self._lib.nmch_engine_init_ms(self._h)

    def launch_info(self) -> dict:
        li = capi.NmchLaunchInfo()
        capi.check(self._lib.nmch_engine_launch_info(self._h, C.byref(li)))
        return {n: getattr(li, n) for n, _ in li._fields_}

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Group:
    """Single-process multi-GPU group (nmch_group_* of the C ABI): paths sharded over n_gpus devices, one
    ncclAllReduce of the partial moments per compute()/explore()."""

    def __init__(self, n_gpus: int, **kw):
        self._lib = capi.load()
        defaults = dict(NTPB=512, NB=512, T=1.0, S_0=1.0, v_0=0.1, r=0.0, k=0.5, rho=-0.7, theta=0.1, sigma=0.3, N=1000,
                        method=METHOD_FE, floor=FLOOR_ABS, rng=RNG_PHILOX, device=-1, n_paths=0, first_path=0, n_local=0,
                        paths_per_thread=0, block_threads=0)
        defaults.update(kw)
        self.params = capi.NmchParams(*[defaults[n] for n, _ in capi.NmchParams._fields_])
        self._h = C.c_void_p()
        capi.check(self._lib.nmch_group_create(C.byref(self.params), n_gpus, C.byref(self._h)))

    def init(self, seed: int = 1234) -> "Group":
        capi.check(self._lib.nmch_group_init(self._h, seed))
        return self

    def set_params(self, k, theta, sigma) -> None:
        capi.check(self._lib.nmch_group_set_params(self._h, k, theta, sigma))

    def compute(self) -> Moments:
        m = capi.NmchMoments()
        capi.check(self._lib.nmch_group_compute(self._h, C.byref(m)))
        return Moments(m.sum_payoff, m.sum_payoff_sq, m.n_paths, m.exec_ms)

    def explore(self, k, theta, sigma):
        k = np.ascontiguousarray(k, np.float32)
        theta = np.ascontiguousarray(theta, np.float32)
        sigma = np.ascontiguousarray(sigma, np.float32)
        out = (capi.NmchMoments * len(k))()
        f32p = C.POINTER(C.c_float)
        capi.check(self._lib.nmch_group_explore(self._h, k.ctypes.data_as(f32p), theta.ctypes.data_as(f32p),
                                                sigma.ctypes.data_as(f32p), len(k), out))
        return [Moments(m.sum_payoff, m.sum_payoff_sq, m.n_paths, m.exec_ms) for m in out]

    def compute_strikes(self, strikes):
        return _strike_call(self._lib.nmch_group_compute_strikes, self._h, strikes, capi.NmchStrikeMoments, _strike_rows)

    def compute_greeks(self, strikes):
        return _strike_call(self._lib.nmch_group_compute_greeks, self._h, strikes, capi.NmchGreekMoments, _greek_rows)

    def compute_sensitivities(self, strikes):
        return _strike_call(self._lib.nmch_group_compute_sensitivities, self._h, strikes, capi.NmchSensitivityMoments,
                            _sensitivity_rows)

    @property
    def size(self) -> int:
        return self._lib.nmch_group_size(self._h)

    @property
    def init_ms(self) -> float:
        return self._lib.nmch_group_init_ms(self._h)

    def finalize(self) -> None:
        if self._h:
            capi.check(self._lib.nmch_group_finalize(self._h))

    def close(self) -> None:
        if self._h:
            self._lib.nmch_group_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
