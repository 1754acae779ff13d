"""Azimuth-averaged phase functions P0(mu, mu0) and P(mu, mu') for the analytic / tabulated families.

Input producer of the hot path (SURVEY.md 8a row a11, 8f rank 1).  Same quadrature as the
reference builders -- 25 azimuth nodes on [0, pi], both half-rings, composite trapezoid, raw
matrix symmetric, then every *column* normalised so that trapz(P[:, n], mu) = 4
(SOS_Aer_phase_func.py:68-292) -- but evaluated as array expressions instead of the reference's
triple Python loop (89-112 s per matrix at N = 1002 there, well under a second here).

Log-normal Mie aerosols (SOS_Aer_phase_func.py:398-753, the reference's 'eva' / 'wildfire' families) need
`miepython`, which the reference does not pin and which is not installed here: family 'mie_lognormal' takes
its tabulated mixture phase function from the host Lorenz-Mie stand-in of mie.py (g = (wavelength, n_re, n_im,
r_m, sigma), e.g. mie.EVA_AEROSOL) and then goes through the same tabulated builder as the FWC cloud.  Callers
with their own Mie code still pass (P0, P) arrays.
"""
from __future__ import annotations

import os

import numpy as np

NB_PHI = 25  # SOS_Aer_phase_func.py:81

_FWC = None


def _fwc_table():
    """The tabulated FWC cloud phase function (data of SOS_Aer_fwc_data.py:3,173)."""
    global _FWC
    if _FWC is None:
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "fwc_table.npz")
        d = np.load(path)
        _FWC = (d["mu_fwc"], d["phase_func_FWC"])
    return _FWC


def phase_table(name, g=None):
    """(cos Theta ascending, values) of a tabulated family: 'fwc', or 'mie_lognormal' with g = (wl, n_re, n_im, r_m, sigma)."""
    name, g = resolve(name, g)
    if name == "fwc":
        return _fwc_table()
    if name == "mie_lognormal":
        from . import mie
        return mie.lognormal_table(*[float(v) for v in g])
    raise ValueError(f"{name!r} is not a tabulated phase function")


TABULATED = ("fwc", "mie_lognormal")


def resolve(name, g=None):
    """The reference's dispatcher names for its two Mie aerosols (phase_func(), SOS_Aer_phase_func.py:12-63: 'eva',
    'wildfire') -> ('mie_lognormal', parameters); every other family is returned unchanged."""
    if name in ("eva", "wildfire"):
        from . import mie
        return "mie_lognormal", (mie.EVA_AEROSOL if name == "eva" else mie.WILDFIRE_AEROSOL)
    return name, g


def _trapz(y, x, axis=-1):
    y = np.asarray(y)
    d = np.diff(x)
    y = np.moveaxis(y, axis, -1)
    return (d * (y[..., 1:] + y[..., :-1]) / 2.0).sum(-1)


def _kernel(name, g):
    if name == "rayleigh":
        return lambda c: 0.75 * (1 + c * c)  # SOS_Aer_phase_func.py:97
    if name == "hg":
        return lambda c: (1 - g * g) / ((1 + g * g - 2 * g * c) ** 1.5)  # :158
    if name in TABULATED:
        xs, ys = phase_table(name, g)

        def interp(c):  # interpolate_fwc_phase, :202-236
            c = np.clip(c, -1, 1)
            i = np.searchsorted(xs, c)
            lo = np.clip(i - 1, 0, len(xs) - 1)
            hi = np.clip(i, 0, len(xs) - 1)
            with np.errstate(all="ignore"):
                w = (c - xs[lo]) / (xs[hi] - xs[lo])
                v = ys[lo] + w * (ys[hi] - ys[lo])
            v = np.where(i == 0, ys[0], v)
            v = np.where(i >= len(xs), ys[-1], v)
            return v
        return interp
    raise ValueError(f"unknown analytic phase function {name!r}")


def phase_P0(name: str, nb_angles: int, mu: np.ndarray, mu0: float, g: float = 0.5) -> np.ndarray:
    """First-order phase function P0(mu, mu0), normalised to trapz(P0, mu) = 2 (:92-105)."""
    name, g = resolve(name, g)
    N = 2 * nb_angles
    mu = np.asarray(mu, dtype=np.float64)
    if name == "iso":
        return np.ones(N)  # :71
    f = _kernel(name, g)
    phi = np.linspace(0, np.pi, NB_PHI)
    cphi = np.cos(0 - phi)
    s = np.sqrt(1 - mu * mu)
    cc = (mu * mu0)[:, None]
    ss = (np.sqrt(1 - mu0 * mu0) * s)[:, None] * cphi[None, :]
    P0 = _trapz(f(-(cc + ss)) + f(-(cc - ss)), phi) / (4 * np.pi)
    return P0 / _trapz(P0, mu) * 2


def phase_P(name: str, nb_angles: int, mu: np.ndarray, g: float = 0.5, block: int = 128) -> np.ndarray:
    """P(mu, mu'): raw matrix symmetric, then every column normalised to trapz = 4 (:112-131)."""
    name, g = resolve(name, g)
    N = 2 * nb_angles
    mu = np.asarray(mu, dtype=np.float64)
    if name == "iso":
        return 2 * np.ones((N, N))  # :74
    f = _kernel(name, g)
    phi = np.linspace(0, np.pi, NB_PHI)
    cphi = np.cos(0 - phi)
    s = np.sqrt(1 - mu * mu)
    P = np.empty((N, N))
    for a in range(0, N, block):
        b = min(N, a + block)
        cmn = mu[:, None] * mu[None, a:b]                       # mu[m]*mu[n]
        smn = (s[None, a:b] * s[:, None])                       # sqrt(1-mu[n]^2)*sqrt(1-mu[m]^2)
        x = smn[:, :, None] * cphi[None, None, :]
        P[:, a:b] = _trapz(f(-(cmn[:, :, None] + x)) + f(-(cmn[:, :, None] - x)), phi) / (2 * np.pi)
    return 4 * P / _trapz(P, mu, axis=0)[None, :]


def phase_matrices(name: str, nb_angles: int, mu: np.ndarray, mu0: float, g: float = 0.5):
    """Return (P0 (N,), P (N, N)) for name in {'iso', 'rayleigh', 'hg', 'fwc', 'mie_lognormal'}."""
    return phase_P0(name, nb_angles, mu, mu0, g), phase_P(name, nb_angles, mu, g)


def mode_vanishes(name: str, m: int) -> bool:
    """True when Fourier mode m of the family is identically zero: isotropic m >= 1, Rayleigh m >= 3 (0.75 (1 + cos^2 Theta)
    is a polynomial of degree 2 in cos(phi)).  The builders return rounding-level values there; solvers use exact zeros."""
    return m >= 1 and (name == "iso" or (name == "rayleigh" and m >= 3))


def azimuth_nodes(n_quad: int, n_modes: int):
    """(phi (n_quad,), table (1 + n_modes, n_quad)) of the mode builders: phi = linspace(0, pi, n_quad), table row 0 =
    cos(0 - phi) (the node cosines of the azimuth-averaged builders), row 1 + m = cos(m phi)."""
    phi = np.linspace(0, np.pi, int(n_quad))
    tab = np.empty((1 + int(n_modes), phi.size))
    tab[0] = np.cos(0 - phi)
    tab[1:] = np.cos(np.arange(int(n_modes))[:, None] * phi[None, :])
    return phi, tab


def _mode_rings(f, cc, x, cm, phi):
    """trapz over phi of cos(m phi) [f(-(cc - x)) + (-1)^m f(-(cc + x))] for every m (leading axis); mode 0 in the
    operation order of phase_P0 / phase_P.  cc: (..., 1), x: (..., n_quad), cm: (K, n_quad)."""
    fb, fa = f(-(cc + x)), f(-(cc - x))
    even, odd = fb + fa, fa - fb
    out = [_trapz(even, phi)]
    for m in range(1, cm.shape[0]):
        out.append(_trapz(cm[m] * (odd if m & 1 else even), phi))
    return np.stack(out)


FAMILY_CODE = {"rayleigh": 0, "hg": 1, "fwc": 2, "mie_lognormal": 2}   # the device's phase families (csrc/phase.cuh)


def exact_norm(name: str, mu: np.ndarray, mu0: float, g=0.5, n_quad: int = 25) -> float:
    """T = trapz_mu(ring_0 / 4 pi): the mode-0 normalisation phase_modes divides the solar modes by at n_quad azimuth nodes
    (at n_quad = 25 that of phase_P0), so that sum_m (2 - delta_m0) P0_m cos(m phi) -> p(cos Theta) / T as K -> infinity."""
    name, g = resolve(name, g)
    f = _kernel(name, g)
    mu = np.asarray(mu, dtype=np.float64)
    phi = np.linspace(0, np.pi, int(n_quad))
    cc = (mu * mu0)[:, None]
    x = (np.sqrt(1 - mu0 * mu0) * np.sqrt(1 - mu * mu))[:, None] * np.cos(0 - phi)[None, :]
    return float(_trapz(_trapz(f(-(cc + x)) + f(-(cc - x)), phi) / (4 * np.pi), mu))


def phase_exact(name: str, nb_angles: int, mu: np.ndarray, mu0: float, phi, g=0.5, n_quad: int = 25) -> np.ndarray:
    """The solar phase vector at the azimuths phi, (n_phi, N): p(cos Theta(mu, mu0, phi)) / T with cos Theta = -mu0 mu +
    sqrt(1 - mu0^2) sqrt(1 - mu^2) cos phi (the convention of phase_modes) and T = exact_norm(..., n_quad): the value the
    series sum_m (2 - delta_m0) P0_m cos(m phi) of phase_modes(..., n_quad) converges to.  Isotropic: ones."""
    name, g = resolve(name, g)
    mu = np.asarray(mu, dtype=np.float64)
    phi = np.atleast_1d(np.asarray(phi, dtype=np.float64))
    if name == "iso":
        return np.ones((phi.size, 2 * nb_angles))
    c = -mu0 * mu[None, :] + np.sqrt(1 - mu0 * mu0) * np.sqrt(1 - mu * mu)[None, :] * np.cos(phi)[:, None]
    return _kernel(name, g)(c) / exact_norm(name, mu, mu0, g, n_quad)


def phase_modes(name: str, nb_angles: int, mu: np.ndarray, n_modes: int, g: float = 0.5, mu0=None, n_quad: int = 25,
                want_P: bool = True):
    """Azimuthal Fourier modes m = 0 .. n_modes-1 of a phase function: (P0_m (K, N) or None without mu0, P_m (K, N, N) or
    None with want_P=False).

    phi is the azimuth of the propagation direction of the scattered light relative to the propagation azimuth of the
    incident light (the solar beam travels along (-mu0, 0): cos Theta = -mu0 mu + sqrt(1 - mu0^2) sqrt(1 - mu^2) cos phi;
    phi = 0 is the forward half-plane, a sensor's relative viewing azimuth is phi + pi).  Mode m integrates the builders'
    integrand over the n_quad nodes of [0, pi] with weight cos(m phi): trapz(cos(m phi) [f(-(cc - x)) + (-1)^m f(-(cc + x))]),
    and every mode is normalised by the column integrals of MODE 0 (P_m[:, n] = 4 R_m[:, n] / trapz(R_0[:, n], mu),
    P0_m = 2 P0raw_m / trapz(P0raw_0, mu)), so that sum_m (2 - delta_m0) P0_m cos(m phi) = c p(cos Theta) with one
    constant c.  Mode 0 is phase_P0 / phase_P at n_quad = 25.  n_quad nodes resolve modes well below n_quad (mode m aliases
    with harmonics 2 (n_quad - 1) +- m)."""
    name, g = resolve(name, g)
    N, K = 2 * nb_angles, int(n_modes)
    mu = np.asarray(mu, dtype=np.float64)
    P0 = P = None
    if name == "iso":
        if mu0 is not None:
            P0 = np.zeros((K, N))
            P0[0] = 1.0
        if want_P:
            P = np.zeros((K, N, N))
            P[0] = 2.0
        return P0, P
    f = _kernel(name, g)
    phi, tab = azimuth_nodes(n_quad, K)
    cphi, cm = tab[0], tab[1:]
    s = np.sqrt(1 - mu * mu)
    if mu0 is not None:
        cc = (mu * mu0)[:, None]
        x = (np.sqrt(1 - mu0 * mu0) * s)[:, None] * cphi[None, :]
        P0 = _mode_rings(f, cc, x, cm, phi) / (4 * np.pi)
        P0 = P0 / _trapz(P0[0], mu) * 2
    if want_P:
        P = np.empty((K, N, N))
        blk = max(1, (1 << 22) // max(1, N * phi.size))
        for a in range(0, N, blk):
            b = min(N, a + blk)
            cmn = mu[:, None] * mu[None, a:b]
            smn = s[None, a:b] * s[:, None]
            x = smn[:, :, None] * cphi[None, None, :]
            P[:, :, a:b] = _mode_rings(f, cmn[:, :, None], x, cm, phi) / (2 * np.pi)
        P = 4 * P / _trapz(P[0], mu, axis=0)[None, None, :]
    return P0, P
