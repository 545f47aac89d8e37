"""Float64 reference of Andersen's QE-M scheme (Andersen 2008, "Efficient simulation of the Heston stochastic volatility
model") on the QE kernel's Philox draws (plain numpy).

The checker of qe_kernel that shares neither its instructions nor its folded arithmetic: the scheme is written from the
paper, and is itself pinned by quadrature of its conditional moments and of the martingale condition
(tests/test_qe64_reference.py).

  Philox4x32-10, counter (step, call, path_lo, path_hi), key (seed_lo, seed_hi): one block per (path, step).
  u(w) = ((w >> 9) + 1/2) 2^-23;  Z_v = sqrt(-2 ln u(x)) sin(a),  Z_s = sqrt(-2 ln u(x)) cos(a),  a = 2 pi (y >> 9) 2^-23;
  U = u(z), the uniform of the exponential branch.
  m = theta + (V - theta) e^{-k dt},  s^2 = V sigma^2 e^{-k dt} (1 - e^{-k dt}) / k + theta sigma^2 (1 - e^{-k dt})^2 / (2k),
  psi = s^2 / m^2.
  psi <= 1.5:  b^2 = 2/psi - 1 + sqrt(2/psi) sqrt(2/psi - 1),  a = m / (1 + b^2),  V' = a (b + Z_v)^2,
               M = exp(A b^2 a / (1 - 2 A a)) / sqrt(1 - 2 A a).
  psi > 1.5:   p = (psi - 1) / (psi + 1),  beta = (1 - p) / m,  V' = 0 if U <= p else ln((1 - p) / (1 - U)) / beta,
               M = p + beta (1 - p) / (beta - A).
  m = 0 (theta = 0 and V = 0): V' = 0 and M = 1, the CIR process is absorbed at zero.
  ln S' = ln S + r dt + K0* + K1 V + K2 V' + sqrt(K3 V + K4 V') Z_s,  K0* = -ln M - (K1 + K3 / 2) V,
  K1 = g1 dt (k rho / sigma - 1/2) - rho / sigma,  K2 = g2 dt (k rho / sigma - 1/2) + rho / sigma,
  K3 = g1 dt (1 - rho^2),  K4 = g2 dt (1 - rho^2),  A = K2 + K4 / 2,  g1 = g2 = 1/2.
  dt = T / N in float64, with the parameters at their float32 values, as the kernel's host fold forms it.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from fe64_reference import philox4x32_10

PSI_C = 1.5
G1 = G2 = 0.5
_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)


def uniform23(w):
    """The kernel's open uniform from the top 23 bits of a word: ((w >> 9) + 1/2) 2^-23, exact in float64."""
    return ((w >> np.uint64(9)).astype(np.float64) + 0.5) * 2.0 ** -23


def draws(x, y, z):
    """(Z_v, Z_s, U) of one Philox block, in float64."""
    rad = np.sqrt(-2.0 * np.log(uniform23(x)))
    ang = (y >> np.uint64(9)).astype(np.float64) * (2.0 * np.pi * 2.0 ** -23)
    return rad * np.sin(ang), rad * np.cos(ang), uniform23(z)


@dataclass
class Coefs:
    e: float            # e^{-k dt}
    dt: float
    k: float
    theta: float
    sigma: float
    K0: float
    K1: float
    K2: float
    K3: float
    K4: float

    @property
    def A(self):
        return self.K2 + 0.5 * self.K4


def coefs(T, k, rho, theta, sigma, N) -> Coefs:
    dt = T / N
    K0 = -rho * k * theta * dt / sigma
    K1 = G1 * dt * (k * rho / sigma - 0.5) - rho / sigma
    K2 = G2 * dt * (k * rho / sigma - 0.5) + rho / sigma
    K3, K4 = G1 * dt * (1.0 - rho * rho), G2 * dt * (1.0 - rho * rho)
    return Coefs(np.exp(-k * dt), dt, k, theta, sigma, K0, K1, K2, K3, K4)


def moments(c: Coefs, V):
    """The conditional mean and variance of the CIR transition over dt, given V."""
    om = -np.expm1(-c.k * c.dt)
    m = c.theta + (V - c.theta) * c.e
    s2 = V * c.sigma ** 2 * c.e * om / c.k + c.theta * c.sigma ** 2 * om * om / (2.0 * c.k)
    return m, s2


def quadratic(psi, m):
    """(a, b) of the psi <= 1.5 branch, V' = a (b + Z)^2."""
    t = 2.0 / psi
    b2 = t - 1.0 + np.sqrt(t) * np.sqrt(t - 1.0)
    return m / (1.0 + b2), np.sqrt(b2)


def exponential(psi, m):
    """(p, beta) of the psi > 1.5 branch: V' = 0 with probability p, else exponential with rate beta."""
    one_p = 2.0 / (psi + 1.0)                # 1 - p without cancellation for large psi
    return 1.0 - one_p, one_p / m


def step(c: Coefs, V, zv, u):
    """One variance step: (V', ln M, psi, existence of M).  Where m = 0 the step is absorbed (V' = 0, ln M = 0)."""
    m, s2 = moments(c, V)
    live = m > 0.0
    mm = np.where(live, m, 1.0)
    psi = np.where(live, s2 / (mm * mm), 0.0)
    quad = psi <= PSI_C
    A = c.A
    with np.errstate(divide="ignore", invalid="ignore"):
        a, b = quadratic(np.where(quad, psi, 1.0), mm)
        d = 1.0 - 2.0 * A * a
        lnM_q = A * b * b * a / d - 0.5 * np.log(d)
        p, beta = exponential(np.where(quad, 2.0, psi), mm)
        v_exp = np.where(u <= p, 0.0, np.log((1.0 - p) / (1.0 - u)) / beta)
        lnM_e = np.log(p + beta * (1.0 - p) / (beta - A))
        Vn = np.where(quad, a * (b + zv) ** 2, v_exp)
    lnM = np.where(quad, lnM_q, lnM_e)
    exists = np.where(quad, d > 0.0, beta > A)
    Vn = np.where(live, Vn, 0.0)
    lnM = np.where(live, lnM, 0.0)
    exists = np.where(live, exists, True)
    return Vn, lnM, np.where(live, psi, np.nan), quad & live, p, exists


def log_increment(c: Coefs, r, V, Vn, lnM, zs):
    """ln S' - ln S of one step: r dt + K0* + K1 V + K2 V' + sqrt(K3 V + K4 V') Z_s."""
    K0s = -lnM - (c.K1 + 0.5 * c.K3) * V
    return r * c.dt + K0s + c.K1 * V + c.K2 * Vn + np.sqrt(c.K3 * V + c.K4 * Vn) * zs


@dataclass
class Paths:
    S: np.ndarray           # S_T
    V: np.ndarray           # V_T
    psi_margin: np.ndarray  # min over steps of |psi - 1.5|: how close a step came to the branch switch
    u_margin: np.ndarray    # min over exponential-branch steps of |U - p|: how close V' came to the point mass
    no_martingale: np.ndarray   # some step had 1 - 2 A a <= 0 or beta <= A: M does not exist there


def qe_paths(T=1.0, S_0=1.0, v_0=0.1, r=0.0, k=0.5, rho=-0.7, theta=0.1, sigma=0.3, N=50, seed=1234, first_path=0,
             n_paths=1024, call=0) -> Paths:
    """Paths [first_path, first_path + n_paths) of the QE pass with call id `call` (the engine's call counter; point i
    of an explore() uses call0 + i)."""
    f32 = np.float32
    T, S0, v0, r, k, rho, theta, sigma = (float(f32(x)) for x in (T, S_0, v_0, r, k, rho, theta, sigma))
    c = coefs(T, k, rho, theta, sigma, N)
    path = np.arange(n_paths, dtype=np.uint64) + np.uint64(first_path)
    plo, phi = path & _LO, path >> _32
    key = (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    lnS = np.full(n_paths, np.log(S0))
    V = np.full(n_paths, v0)
    psi_margin = np.full(n_paths, np.inf)
    u_margin = np.full(n_paths, np.inf)
    bad = np.zeros(n_paths, bool)
    for n in range(N):
        x, y, z, _ = philox4x32_10((n, call & 0xFFFFFFFF, plo, phi), key)
        zv, zs, u = draws(x, y, z)
        Vn, lnM, psi, quad, p, exists = step(c, V, zv, u)
        psi_margin = np.minimum(psi_margin, np.where(np.isnan(psi), np.inf, np.abs(psi - PSI_C)))
        u_margin = np.minimum(u_margin, np.where(quad | np.isnan(psi), np.inf, np.abs(u - p)))
        bad |= ~exists
        lnS = lnS + log_increment(c, r, V, Vn, lnM, zs)
        V = Vn
    return Paths(np.exp(lnS), V, psi_margin, u_margin, bad)
