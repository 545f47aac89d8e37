"""Float64 reference of the native FE step on cuRAND's Philox stream, with the pathwise tangent in v_0 (plain numpy).

The checker of compute_greeks() and compute_strikes() that shares neither the product's instructions nor its
derivation: the step is written from the model, the tangent is carried by forward-mode differentiation of that step
and is itself checked against a central finite difference of the float64 paths (tests/test_fe64_reference.py).

  Philox4x32-10, counter (blk_lo, blk_hi, path_lo, path_hi), key (seed_lo, seed_hi).  Step n of a pass that starts
  w0 words into the stream uses block (w0/2 + n) >> 1, words (x, y) when w0/2 + n is even and (z, w) when it is odd
  (curand_normal2 on curand_init(seed, path, w0)).
  u = x 2^-32 + 2^-33,  angle = y 2 pi 2^-32,  Z1 = sqrt(-2 ln u) sin(angle),  Z2 = sqrt(-2 ln u) cos(angle)
  S' = S (1 + r dt + sqrt(V dt) (rho Z1 + sqrt(1 - rho^2) Z2))
  V' = g(V + kappa (theta - V) dt + sigma sqrt(V dt) Z1),   g = |.| or (.)+,   S' uses V before its update
  dt = float32(T) / float32(N) in float32, as the reference forms it; everything else in float64.
  A = dV/dv_0, B = dS/dv_0 (A_0 = 1, B_0 = 0).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)

FLOOR_ABS, FLOOR_PLUS = 0, 1
# the order of the sums of one strike, in compute_greeks' raw layout
SUMS = ("payoff", "payoff_sq", "delta", "itm", "vega", "vega_sq")


def philox4x32_10(ctr, key):
    """Philox4x32-10 of counters (c0, c1, c2, c3) (each a scalar or an array, broadcast) under key (k0, k1).
    Returns the four output words as uint64 arrays holding 32-bit values."""
    c0, c1, c2, c3 = np.broadcast_arrays(*(np.asarray(c, dtype=np.uint64) for c in ctr))
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for _ in range(10):
        p0 = _M0 * c0                                   # 32 x 32 -> 64 bits: exact in uint64
        p1 = _M1 * c2
        c0, c1, c2, c3 = (p1 >> _32) ^ c1 ^ np.uint64(k0), p1 & _LO, (p0 >> _32) ^ c3 ^ np.uint64(k1), p0 & _LO
        k0 = (k0 + _W0) & 0xFFFFFFFF
        k1 = (k1 + _W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


def normals(x, y):
    """cuRAND's Box-Muller pair from two words, in float64: (Z1, Z2) = sqrt(-2 ln u) (sin, cos)(angle)."""
    u = x.astype(np.float64) * 2.0 ** -32 + 2.0 ** -33
    ang = y.astype(np.float64) * (2.0 * np.pi * 2.0 ** -32)
    rad = np.sqrt(-2.0 * np.log(u))
    return rad * np.sin(ang), rad * np.cos(ang)


@dataclass
class Paths:
    S: np.ndarray           # S_T
    V: np.ndarray           # V_T
    A: np.ndarray           # dV_T / dv_0
    B: np.ndarray           # dS_T / dv_0
    margin: np.ndarray      # min over steps of |pre-floor V'| / |sigma sqrt(V dt) Z1|: how close the path came to the kink


def fe_paths(T=1.0, S_0=1.0, v_0=0.1, r=0.0, k=0.5, rho=-0.7, theta=0.1, sigma=0.3, N=1000, floor=FLOOR_ABS,
             seed=1234, first_path=0, n_paths=1024, offset=0, v0_shift=0.0) -> Paths:
    """Paths [first_path, first_path + n_paths) of one pass that starts `offset` 32-bit words into every path's stream
    (offset even: a pass consumes two words per step).  The parameters are taken at their float32 values, as the
    kernels see them; v0_shift is added to v_0 after that rounding (a finite difference in v_0 below float32's ulp)."""
    if offset % 2:
        raise ValueError("offset must be an even number of words")
    f32 = np.float32
    dt = float(f32(T) / f32(N))
    S0, v0, r, k, rho, theta, sigma = (float(f32(x)) for x in (S_0, v_0, r, k, rho, theta, sigma))
    v0 += v0_shift
    crho = np.sqrt(1.0 - rho * rho)
    path = np.arange(n_paths, dtype=np.uint64) + np.uint64(first_path)
    plo, phi = path & _LO, path >> _32
    key = (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    S = np.full(n_paths, S0)
    V = np.full(n_paths, v0)
    A = np.ones(n_paths)
    B = np.zeros(n_paths)
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
            dsq = np.where(V > 0.0, sq * A / (2.0 * V), 0.0)        # d sqrt(V dt) / dv_0; V = 0 is parked with A = 0
        zs = rho * z1 + crho * z2
        growth = 1.0 + r * dt + sq * zs
        B = B * growth + S * zs * dsq
        S = S * growth
        noise = sigma * sq * z1
        vpre = V + k * (theta - V) * dt + noise
        apre = A * (1.0 - k * dt) + sigma * z1 * dsq
        with np.errstate(divide="ignore", invalid="ignore"):
            margin = np.minimum(margin, np.where(noise != 0.0, np.abs(vpre) / np.abs(noise), np.inf))
        if floor == FLOOR_ABS:
            A = np.where(vpre < 0.0, -apre, apre)
            V = np.abs(vpre)
        else:
            A = np.where(vpre > 0.0, apre, 0.0)
            V = np.maximum(vpre, 0.0)
    return Paths(S, V, A, B, margin)


def strike_fold_bounds(S, B, K, S_0, delta):
    """The six sums of one strike (SUMS) over the reference paths, as intervals.

    A path with |S - K| <= delta max(|K|, S) (delta: the per-path relative tolerance of S) may fall on either side of
    the strike in the kernel under test, so it widens the interval by its whole in-the-money contribution.  Returns
    (lo, hi, scale): scale is the sum of |contribution| over every path that may be in the money, the size against
    which a relative tolerance for the per-path errors of S and B is set."""
    S = np.asarray(S, np.float64)
    B = np.asarray(B, np.float64)
    K = float(np.float32(K))
    band = delta * np.maximum(abs(K), np.abs(S))
    amb = np.abs(S - K) <= band
    itm = (S > K) & ~amb
    pay = np.where(amb, np.abs(S - K) + band, np.maximum(S - K, 0.0))
    contrib = np.stack([pay, pay * pay, S / float(np.float32(S_0)), np.ones_like(S), B, B * B])
    sure = contrib[:, itm].sum(axis=1)
    lo = sure + np.minimum(contrib[:, amb], 0.0).sum(axis=1)
    hi = sure + np.maximum(contrib[:, amb], 0.0).sum(axis=1)
    scale = np.abs(contrib[:, itm | amb]).sum(axis=1)
    return lo, hi, scale
