"""Ross-Li bidirectional ground reflectance: the kernels, their azimuthal Fourier modes on the mu grid (NumPy reference).

rho(mu_i, mu_v, psi) = f_iso + f_vol K_vol + f_geo K_geo, the kernel-driven model of the MODIS / VIIRS BRDF-albedo products:
RossThick and LiSparse-Reciprocal after Lucht, Schaaf & Strahler (2000), with h/b = 2 and b/r = 1.  psi is the Ross-Li
relative azimuth, with the backscatter hot spot at psi = 0.

The engine's phi is the PROPAGATION azimuth relative to the incident light's (azimuth module), so psi = phi - pi and the
hot spot of the radiance reflected from the solar beam sits at engine phi = pi.  In that convention the modes are

    rho_m(mu, mu') = (1/pi) int_0^pi rho(mu, mu', phi - pi) cos(m phi) dphi = (-1)^m rho_m^{Ross-Li},

with rho = rho_0 + 2 sum_{m >= 1} rho_m cos(m phi), the normalisation of the radiance modes; they are integrated with the
trapezoid rule on BRDF_NODES nodes on [0, pi].  Both zenith arguments are clamped to mu >= BRDF_MU_MIN = cos 85 deg (a model
choice: K_geo grows like sec(theta), so grazing columns of the grid would reflect hundreds of times their nadir radiance).
csrc/brdf.cuh builds the same matrices on the device (SosEngine.build_brdf_modes); these functions are the reference the
tests compare against and build the per-scenario beam vectors on the host.
"""
from __future__ import annotations

import numpy as np

BRDF_NODES = 361                       # azimuth nodes of the mode integrals, whatever the phase builder's n_quad
BRDF_MU_MIN = float(np.cos(np.radians(85.0)))
KERNELS = ("vol", "geo")


def rossli_kernels(mu_i, mu_v, psi):
    """(K_vol, K_geo) at illumination / view zenith cosines mu_i, mu_v (> 0) and Ross-Li relative azimuth psi (broadcast)."""
    mi, mv, psi = np.broadcast_arrays(np.asarray(mu_i, dtype=np.float64), np.asarray(mu_v, dtype=np.float64),
                                      np.asarray(psi, dtype=np.float64))
    cp = np.cos(psi)
    si, sv = np.sqrt((1 - mi) * (1 + mi)), np.sqrt((1 - mv) * (1 + mv))
    cx = np.clip(mi * mv + si * sv * cp, -1.0, 1.0)
    xi = np.arccos(cx)
    k_vol = ((np.pi / 2 - xi) * cx + np.sin(xi)) / (mi + mv) - np.pi / 4
    ti, tv, seci, secv = si / mi, sv / mv, 1 / mi, 1 / mv
    d2 = (ti - tv) ** 2 + 2 * ti * tv * (1 - cp)   # D^2 without cancellation at the hot spot (1 - cp is exact)
    ct = np.clip(2 * np.sqrt(d2 + (ti * tv) ** 2 * ((1 - cp) * (1 + cp))) / (seci + secv), -1.0, 1.0)
    t = np.arccos(ct)
    overlap = (t - np.sin(t) * ct) * (seci + secv) / np.pi
    k_geo = overlap - (seci + secv) + 0.5 * (1 + cx) * (seci * secv)   # (every operation symmetric: exactly reciprocal)
    return k_vol, k_geo


def node_table(n_quad: int, n_modes: int):
    """(phi (n_quad,), table (1 + n_modes, n_quad)): phi = linspace(0, pi, n_quad); table row 0 = cos(phi - pi) (the
    kernels' cos psi), row 1 + m = cos(m phi).  What sos_build_brdf_modes takes."""
    phi = np.linspace(0, np.pi, int(n_quad))
    tab = np.empty((1 + int(n_modes), phi.size))
    tab[0] = np.cos(phi - np.pi)
    tab[1:] = np.cos(np.arange(int(n_modes))[:, None] * phi[None, :])
    return phi, tab


def _mode_weights(n_modes: int, n_quad: int):
    """(n_quad, n_modes): trapezoid weight of node k times cos(m phi_k) / pi, and the nodes phi_k."""
    phi, tab = node_table(n_quad, n_modes)
    w = np.empty(phi.size)
    w[1:-1] = 0.5 * (phi[2:] - phi[:-2])
    w[0], w[-1] = 0.5 * (phi[1] - phi[0]), 0.5 * (phi[-1] - phi[-2])
    return (w[:, None] * tab[1:].T) / np.pi, phi


def _modes(mu_a, mu_b, n_modes, n_quad):
    """Both kernels' modes (2, n_modes, *shape) at the clamped cosines mu_a, mu_b (arrays of one shape)."""
    wc, phi = _mode_weights(n_modes, n_quad)
    a = np.maximum(mu_a, BRDF_MU_MIN)[..., None]
    b = np.maximum(mu_b, BRDF_MU_MIN)[..., None]
    kv, kg = rossli_kernels(a, b, phi - np.pi)
    return np.stack([np.moveaxis(kv @ wc, -1, 0), np.moveaxis(kg @ wc, -1, 0)])


def _check(kernel):
    if kernel not in KERNELS:
        raise ValueError(f"kernel must be one of {KERNELS}, not {kernel!r}")
    return KERNELS.index(kernel)


def brdf_modes(kernel: str, M: int, mu: np.ndarray, n_modes: int, n_quad: int = BRDF_NODES) -> np.ndarray:
    """Modes of one kernel ('vol' or 'geo') on the grid: (n_modes, M-1, M), element [m][i][c] = rho_m(mu[M+1+i], |mu[c]|)
    for the upward columns i and the downward columns c (engine convention, clamped)."""
    k = _check(kernel)
    mu = np.asarray(mu, dtype=np.float64)
    up, down = mu[M + 1: 2 * M], np.abs(mu[:M])
    out = np.empty((int(n_modes), M - 1, M))
    for c in range(M):   # one downward column at a time: (M-1) x n_quad kernel values
        out[:, :, c] = _modes(up, np.full(M - 1, down[c]), n_modes, n_quad)[k]
    return out


def brdf_beam(kernel: str, M: int, mu: np.ndarray, mu0: float, n_modes: int, n_quad: int = BRDF_NODES) -> np.ndarray:
    """Modes of one kernel for the solar beam: (n_modes, M-1), element [m][i] = rho_m(mu[M+1+i], mu0)."""
    k = _check(kernel)
    up = np.asarray(mu, dtype=np.float64)[M + 1: 2 * M]
    return _modes(up, np.full(M - 1, float(mu0)), n_modes, n_quad)[k]


def brdf_synthesis(modes: np.ndarray, phi) -> np.ndarray:
    """rho_0 + 2 sum_{m >= 1} rho_m cos(m phi) for modes (n_modes, ...) at the engine azimuths phi: (len(phi), ...)."""
    modes = np.asarray(modes)
    phi = np.atleast_1d(np.asarray(phi, dtype=np.float64))
    w = 2.0 * np.cos(np.arange(modes.shape[0])[None, :] * phi[:, None])
    w[:, 0] = 1.0
    return np.tensordot(w, modes, axes=(1, 0))
