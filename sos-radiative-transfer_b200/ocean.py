"""Wind-roughened ocean: Cox-Munk sun glint, its azimuthal Fourier modes on the mu grid (NumPy reference).

surface='ocean': rho(mu_i, mu_v, phi) = grd_alb + rho_glint(mu_i, mu_v, phi; W, n), both in reflectance-factor units.  grd_alb
is the isotropic part (whitecaps plus water-leaving light, chosen by the caller) and the 'lambert_diffuse' coupling unchanged;

    rho_glint = r(omega) exp(-tan^2 theta_n / sigma^2) S / (4 sigma^2 mu_i mu_v mu_n^4)

with the isotropic slope variance of Cox & Munk (1954), sigma^2 = 0.003 + 0.00512 W (W the wind speed in m/s), r the
unpolarised Fresnel reflectance at the local incidence angle omega for the relative refractive index n,
cos 2 omega = mu_i mu_v - sqrt(1 - mu_i^2) sqrt(1 - mu_v^2) cos phi, the facet tilt mu_n = (mu_i + mu_v) / (2 cos omega) and
Smith shadowing S = 1 / (1 + Lambda(mu_i) + Lambda(mu_v)), Lambda(mu) = (e^{-nu^2} / (nu sqrt(pi)) - erfc nu) / 2,
nu = mu / (sigma sqrt(1 - mu^2)).  Shadowing keeps the reflectance finite at grazing angles, so no mu clamp is needed.

phi is the engine's PROPAGATION azimuth relative to the incident light's (azimuth module): the glint sits at phi = 0, the
forward direction (the Ross-Li hot spot is at phi = pi).  The modes are rho_m = (1/pi) int_0^pi rho cos(m phi) dphi on
brdf.BRDF_NODES trapezoid nodes, the normalisation of brdf.py.  The glint lobe is narrow in azimuth at low wind, so a
64-mode series cannot reproduce it there (about 10 % of the peak at W = 1 m/s); solve_azimuthal adds the once-reflected
direct beam in closed form (sos_glint_correction).  csrc/glint.cuh evaluates the same reflectance on the device; these
functions are the reference the tests compare against and build the per-scenario beam vectors on the host.
"""
from __future__ import annotations

import math

import numpy as np

from .brdf import BRDF_NODES, _mode_weights

OCEAN_INDEX = 1.34   # relative refractive index of sea water in the visible
_erfc = np.vectorize(math.erfc, otypes=[np.float64])


def slope_variance(wind_speed):
    """Isotropic Cox-Munk slope variance sigma^2 = 0.003 + 0.00512 W (W in m/s)."""
    return 0.003 + 0.00512 * np.asarray(wind_speed, dtype=np.float64)


def fresnel(cos_w, n):
    """Unpolarised Fresnel reflectance at incidence cosine cos_w for the relative refractive index n > 1."""
    ci = np.asarray(cos_w, dtype=np.float64)
    ct = np.sqrt(1.0 - (1.0 - ci * ci) / (n * n))
    rs = (ci - n * ct) / (ci + n * ct)
    rp = (n * ci - ct) / (n * ci + ct)
    return 0.5 * (rs * rs + rp * rp)


def smith_lambda(mu, sigma):
    """Smith's Lambda(mu) for slope standard deviation sigma; Lambda(1) = 0 exactly."""
    mu = np.asarray(mu, dtype=np.float64)
    out = np.zeros(np.broadcast(mu, sigma).shape)
    lt = np.broadcast_to(mu < 1.0, out.shape)
    m = np.broadcast_to(mu, out.shape)[lt]
    s = np.broadcast_to(sigma, out.shape)[lt]
    nu = m / (s * np.sqrt((1.0 - m) * (1.0 + m)))
    out[lt] = 0.5 * (np.exp(-nu * nu) / (nu * np.sqrt(np.pi)) - _erfc(nu))
    return out


def _glint(mi, mv, cphi, sigma2, n, S):
    """rho_glint with the shadowing factor S given; the operations of csrc/glint.cuh, symmetric in (mi, mv).
    D = 4 cos^2 omega - (mi + mv)^2 = (s_i - s_v)^2 + 2 s_i s_v (1 - cos phi) has no cancellation near the specular direction:
    mu_n^2 = (mi + mv)^2 / ((mi + mv)^2 + D), tan^2 theta_n = D / (mi + mv)^2."""
    si, sv = np.sqrt((1.0 - mi) * (1.0 + mi)), np.sqrt((1.0 - mv) * (1.0 + mv))
    D = (si - sv) * (si - sv) + 2.0 * (si * sv) * (1.0 - cphi)
    sum2 = (mi + mv) * (mi + mv)
    q = sum2 + D
    mn2 = sum2 / q
    return fresnel(0.5 * np.sqrt(q), n) * np.exp(-(D / sum2) / sigma2) * S / (4.0 * sigma2 * (mi * mv) * (mn2 * mn2))


def _shadowing(mi, mv, sigma):
    return 1.0 / (1.0 + (smith_lambda(mi, sigma) + smith_lambda(mv, sigma)))


def cox_munk(mu_i, mu_v, phi, wind_speed, n=OCEAN_INDEX):
    """rho_glint at zenith cosines mu_i, mu_v in (0, 1] and engine azimuth phi (glint at phi = 0), broadcast."""
    mi, mv, phi = np.broadcast_arrays(np.asarray(mu_i, dtype=np.float64), np.asarray(mu_v, dtype=np.float64),
                                      np.asarray(phi, dtype=np.float64))
    s2 = slope_variance(wind_speed)
    return _glint(mi, mv, np.cos(phi), s2, n, _shadowing(mi, mv, np.sqrt(s2)))


def _modes(mu_a, mu_b, W, n, n_modes, n_quad):
    """Glint modes (n_modes, *shape) at the cosines mu_a > 0, mu_b >= 0 (one shape); entries with mu_b = 0 are 0."""
    wc, phi = _mode_weights(n_modes, n_quad)
    s2 = float(slope_variance(W))
    a = np.asarray(mu_a, dtype=np.float64)
    b = np.asarray(mu_b, dtype=np.float64)
    out = np.zeros((int(n_modes),) + a.shape)
    live = b > 0
    a, b = a[live][:, None], b[live][:, None]
    rho = _glint(a, b, np.cos(phi)[None, :], s2, n, _shadowing(a, b, np.sqrt(s2)))
    out[:, live] = (rho @ wc).T
    return out


def glint_modes(M: int, mu: np.ndarray, W: float, n: float = OCEAN_INDEX, n_modes: int = 1,
                n_quad: int = BRDF_NODES) -> np.ndarray:
    """Glint modes on the grid: (n_modes, M-1, M), element [m][i][c] = rho_m(mu[M+1+i], |mu[c]|) for the upward columns i
    and the downward columns c (column M-1, mu = 0-, is 0): the layout of brdf.brdf_modes."""
    mu = np.asarray(mu, dtype=np.float64)
    up, down = mu[M + 1: 2 * M], np.abs(mu[:M])
    out = np.empty((int(n_modes), M - 1, M))
    for c in range(M):   # one downward column at a time: (M-1) x n_quad reflectances
        out[:, :, c] = _modes(up, np.full(M - 1, down[c]), W, n, n_modes, n_quad)
    return out


def glint_beam(M: int, mu: np.ndarray, mu0: float, W: float, n: float = OCEAN_INDEX, n_modes: int = 1,
               n_quad: int = BRDF_NODES) -> np.ndarray:
    """Glint modes for the solar beam: (n_modes, M-1), element [m][i] = rho_m(mu[M+1+i], mu0)."""
    up = np.asarray(mu, dtype=np.float64)[M + 1: 2 * M]
    return _modes(up, np.full(M - 1, float(mu0)), W, n, n_modes, n_quad)
