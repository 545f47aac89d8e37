"""Float64 reference of the native FE step with the pathwise tangent in all five Heston parameters (plain numpy).

The checker of compute_sensitivities(): the same paths as fe64_reference.fe_paths (the same Philox words, cuRAND's
Box-Muller pair and the step written from the model, all in float64), carrying dS/dp and dV/dp for
p in DIRS = (v_0, kappa, theta, sigma, rho) by forward-mode differentiation of that step.  It shares no derivation with
the product's folded-constant step (fe_step.cuh); each direction is itself checked against a central finite difference
of the float64 paths (tests/test_fe64_sensitivities.py), and the v_0 direction against fe64_reference's tangent.

  S' = S (1 + r dt + sqrt(V dt) zs),   zs = rho Z1 + sqrt(1 - rho^2) Z2
  V' = g(V + kappa (theta - V) dt + sigma sqrt(V dt) Z1),   g = |.| or (.)+,   S' uses V before its update
  d sqrt(V dt) = sqrt(V dt) dV / (2V)  (taken as 0 at V = 0: the floor parked the path and zeroed dV in that step),
  d zs / d rho = Z1 - rho / sqrt(1 - rho^2) Z2,  d drift / d kappa = (theta - V) dt,  d drift / d theta = kappa dt,
  d noise / d sigma = sqrt(V dt) Z1;  dV_0 / dv_0 = 1, every other initial tangent 0.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from fe64_reference import FLOOR_ABS, FLOOR_PLUS, normals, philox4x32_10, strike_fold_bounds  # noqa: F401

_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)

# the directions, in the order of compute_sensitivities (NMCH_SENS_*)
DIRS = ("v0", "kappa", "theta", "sigma", "rho")


@dataclass
class SensPaths:
    S: np.ndarray           # S_T
    V: np.ndarray           # V_T
    dS: np.ndarray          # (5, n): dS_T / dp for p in DIRS
    dV: np.ndarray          # (5, n): dV_T / dp for p in DIRS (the rho row is 0: V does not depend on rho)
    margin: np.ndarray      # min over steps of |pre-floor V'| / |sigma sqrt(V dt) Z1|, as fe64_reference.Paths.margin


def fe_paths(T=1.0, S_0=1.0, v_0=0.1, r=0.0, k=0.5, rho=-0.7, theta=0.1, sigma=0.3, N=1000, floor=FLOOR_ABS,
             seed=1234, first_path=0, n_paths=1024, offset=0, v0_shift=0.0, k_shift=0.0, theta_shift=0.0,
             sigma_shift=0.0, rho_shift=0.0) -> SensPaths:
    """Paths [first_path, first_path + n_paths) of one pass that starts `offset` 32-bit words into every path's stream,
    as fe64_reference.fe_paths.  The parameters are taken at their float32 values, as the kernels see them; each *_shift
    is added to its parameter after that rounding (a finite difference below float32's ulp)."""
    if offset % 2:
        raise ValueError("offset must be an even number of words")
    f32 = np.float32
    dt = float(f32(T) / f32(N))
    S0, v0, r, k, rho, theta, sigma = (float(f32(x)) for x in (S_0, v_0, r, k, rho, theta, sigma))
    v0 += v0_shift
    k += k_shift
    theta += theta_shift
    sigma += sigma_shift
    rho += rho_shift
    crho = np.sqrt(1.0 - rho * rho)
    path = np.arange(n_paths, dtype=np.uint64) + np.uint64(first_path)
    plo, phi = path & _LO, path >> _32
    key = (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    S = np.full(n_paths, S0)
    V = np.full(n_paths, v0)
    dS = np.zeros((5, n_paths))
    dV = np.zeros((5, n_paths))
    dV[0] = 1.0
    unit = np.eye(5)[:, :, None]                          # unit[d]: 1 in row d, shape (5, 1) after indexing
    margin = np.full(n_paths, np.inf)
    words, cached = None, None
    for n in range(N):
        pair = offset // 2 + n
        blk = pair >> 1
        if blk != cached:
            words = philox4x32_10((blk & 0xFFFFFFFF, blk >> 32, plo, phi), key)
            cached = blk
        z1, z2 = normals(*((words[0], words[1]) if pair % 2 == 0 else (words[2], words[3])))
        sq = np.sqrt(V * dt)
        with np.errstate(divide="ignore", invalid="ignore"):
            dsq = np.where(V > 0.0, sq * dV / (2.0 * V), 0.0)
        zs = rho * z1 + crho * z2
        dzs = np.zeros((5, n_paths))
        dzs[4] = z1 - rho / crho * z2
        growth = 1.0 + r * dt + sq * zs
        dS = dS * growth + S * (dsq * zs + sq * dzs)
        S = S * growth
        noise = sigma * sq * z1
        vpre = V + k * (theta - V) * dt + noise
        dvpre = (dV * (1.0 - k * dt) + unit[1] * ((theta - V) * dt) + unit[2] * (k * dt) + unit[3] * (sq * z1)
                 + sigma * z1 * dsq)
        with np.errstate(divide="ignore", invalid="ignore"):
            margin = np.minimum(margin, np.where(noise != 0.0, np.abs(vpre) / np.abs(noise), np.inf))
        if floor == FLOOR_ABS:
            dV = np.where(vpre < 0.0, -dvpre, dvpre)
            V = np.abs(vpre)
        else:
            dV = np.where(vpre > 0.0, dvpre, 0.0)
            V = np.maximum(vpre, 0.0)
    return SensPaths(S, V, dS, dV, margin)
