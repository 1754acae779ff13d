"""Exact single scattering of azimuth-resolved radiance: phase.phase_exact, the closed-form correction of the first order's
truncated Fourier series (sos_single_scatter_correction) and solve_azimuthal(..., single_scatter='exact').

The NumPy reference of the correction is the oracle's closed-form first order on the difference of the solar phase vectors,
dP0(mu, phi) = p(cos Theta) / T - sum_{m < K} (2 - delta_m0) P0_m(mu) cos(m phi), with the scenario's own ground over a
specular (or black) ground and grd_alb = 0 over the diffuse ones.
"""
import dataclasses
from importlib import import_module

import numpy as np
import pytest

from conftest import relmax

import sos_b200 as sos

PH = import_module("sos-radiative-transfer_b200.phase")
AZ = import_module("sos-radiative-transfer_b200.azimuth")

M_SMALL, L_SMALL = 41, 120
DIFFUSE = ("lambert_diffuse", "rossli", "ocean")


@pytest.fixture(scope="module")
def so():
    import sos_oracle
    return sos_oracle


def small(**kw):
    base = dict(nb_layers=L_SMALL, nb_angles=M_SMALL, tauStar_atm=0.124, tauStar_aer=0.12, grd_alb=0.3, alb_aer=0.97,
                atm_phase=("rayleigh", 0.5), aer_phase=("hg", 0.5), surface="specular")
    base.update(kw)
    return sos.Scenario(**base)


def oracle_scenario(so, sc, ground=True):
    """The oracle's scenario; ground=False: grd_alb = 0 (no mirror term, no upward carry)."""
    osc = so.Scenario(**{f.name: getattr(sc, f.name) for f in dataclasses.fields(so.Scenario)})
    return osc if ground else dataclasses.replace(osc, grd_alb=0.0)


def series_vectors(spec, M, mu, mu0, K, n_quad):
    """The (K, N) solar vectors solve_azimuthal sums: mode 0 = phase_P0 (the base solve), m >= 1 = phase_modes at n_quad
    nodes, exact zeros for a vanishing mode."""
    name, g = PH.resolve(spec[0], spec[1])
    out = np.zeros((K, 2 * M))
    out[0] = sos.phase_P0(name, M, mu, mu0, g)
    if K > 1 and name != "iso":
        P0m, _ = sos.phase_modes(name, M, mu, K, g, mu0=mu0, n_quad=n_quad, want_P=False)
        for m in range(1, K):
            if not PH.mode_vanishes(name, m):
                out[m] = P0m[m]
    return out


def delta_p0(spec, M, mu, mu0, K, n_quad, phi):
    """(n_phi, N): p(cos Theta) / T minus the K-term series; 0 for an isotropic phase function."""
    name, g = PH.resolve(spec[0], spec[1])
    if name == "iso":
        return np.zeros((np.size(phi), 2 * M))
    w = np.cos(np.arange(K)[None, :] * np.atleast_1d(phi)[:, None]) * np.where(np.arange(K) == 0, 1.0, 2.0)[None, :]
    return PH.phase_exact(name, M, mu, mu0, phi, g, n_quad) - w @ series_vectors(spec, M, mu, mu0, K, n_quad)


def reference_correction(so, sc, phi, K, n_quad, rows):
    """(n_rows, n_phi, N): the closed-form first order of dP0 at every azimuth (the NumPy restatement of the device)."""
    osc = oracle_scenario(so, sc, ground=sc.surface not in DIFFUSE)
    tau, _, iu, idn = osc.geometry()
    mu = so.mu_grid(sc.nb_angles)
    da = delta_p0(sc.atm_phase, sc.nb_angles, mu, sc.mu0, K, n_quad, phi)
    de = delta_p0(sc.aer_phase, sc.nb_angles, mu, sc.mu0, K, n_quad, phi)
    return np.stack([so.first_order_regions(osc, tau, mu, iu, idn, da[p], de[p])[list(rows)] for p in range(len(phi))], axis=1)


def oracle_mode(so, sc, P0a, Pa, P0e, Pe, n):
    """The oracle's three-region order loop on one mode's operands for exactly n orders (no ratio test)."""
    osc = oracle_scenario(so, sc)
    tau, _, iu, idn = osc.geometry()
    mu = so.mu_grid(sc.nb_angles)
    I1 = so.first_order_regions(osc, tau, mu, iu, idn, P0a, P0e)
    lay = so.driver_layout(osc, tau, mu, iu, idn)
    dtau_aer = sc.tauStar_aer / (idn + 1 - iu)
    dtau_atm = sc.tauStar_atm / sc.nb_layers
    f_atm, f_aer = dtau_atm / (dtau_atm + dtau_aer), dtau_aer / (dtau_atm + dtau_aer)
    A_atm = so.contraction_matrix(Pa, mu, sc.alb_atm)
    A_mix = f_atm * A_atm + f_aer * so.contraction_matrix(Pe, mu, sc.alb_aer)
    I, In = I1.copy(), I1
    for _ in range(n - 1):
        J = In @ A_atm
        J[iu: idn + 1] = In[iu: idn + 1] @ A_mix
        In = so.order_sweeps(lay, J, method="recurrence")
        I = I + In
    return I


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name,g,K,n_quad,tol", [("rayleigh", 0.5, 3, 25, 1e-14), ("hg", 0.5, 64, 361, 1e-8)])
def test_phase_exact_is_the_limit_of_the_series(name, g, K, n_quad, tol):
    mu, mu0 = sos.mu_grid(M_SMALL), 0.6
    phi = np.linspace(0, 2 * np.pi, 37)
    P0m, _ = sos.phase_modes(name, M_SMALL, mu, K, g, mu0=mu0, n_quad=n_quad, want_P=False)
    syn = P0m[0][None, :] + 2 * np.einsum("kn,kp->pn", P0m[1:], np.cos(np.arange(1, K)[:, None] * phi[None, :]))
    exact = sos.phase_exact(name, M_SMALL, mu, mu0, phi, g, n_quad)
    assert exact.shape == (phi.size, 2 * M_SMALL)
    assert relmax(syn, exact) <= tol


def test_phase_exact_isotropic_and_base_normalisation():
    mu = sos.mu_grid(M_SMALL)
    assert np.array_equal(sos.phase_exact("iso", M_SMALL, mu, 0.5, [0.0, 1.0, 2.0]), np.ones((3, 2 * M_SMALL)))
    # at 25 nodes T is the base solve's phase_P0 normalisation: the azimuth average of p / T is phase_P0
    phi = np.linspace(0, np.pi, 25)
    avg = PH._trapz(sos.phase_exact("hg", M_SMALL, mu, 0.6, phi, 0.7, 25).T, phi) / np.pi
    assert relmax(avg, sos.phase_P0("hg", M_SMALL, mu, 0.6, 0.7)) <= 1e-14


@pytest.mark.parametrize("surface,kw", [("specular", dict(grd_alb=0.3)), ("specular", dict(grd_alb=0.0)),
                                        ("lambert_diffuse", dict(grd_alb=0.3))])
def test_reference_correction_is_linear(so, surface, kw):
    """D[p/T - series] = D[p/T] - D[series]: the correction turns the first order of the series into the exact one."""
    sc = small(surface=surface, aer_phase=("hg", 0.8), mu0=0.45, **kw)
    K, nq, rows = 5, 25, list(range(L_SMALL))
    phi = np.array([0.0, 0.3, np.pi])
    corr = reference_correction(so, sc, phi, K, nq, rows)
    osc = oracle_scenario(so, sc, ground=surface not in DIFFUSE)
    tau, _, iu, idn = osc.geometry()
    mu = so.mu_grid(M_SMALL)
    w = np.cos(np.arange(K)[None, :] * phi[:, None]) * np.where(np.arange(K) == 0, 1.0, 2.0)[None, :]
    for p in range(phi.size):
        ex = [PH.phase_exact(s[0], M_SMALL, mu, sc.mu0, phi[p], s[1], nq)[0] for s in (sc.atm_phase, sc.aer_phase)]
        ser = [w[p] @ series_vectors(s, M_SMALL, mu, sc.mu0, K, nq) for s in (sc.atm_phase, sc.aer_phase)]
        want = so.first_order_regions(osc, tau, mu, iu, idn, *ex) - so.first_order_regions(osc, tau, mu, iu, idn, *ser)
        assert relmax(corr[:, p], want) <= 1e-12, p
    iso = small(surface=surface, atm_phase=("iso", 0.0), aer_phase=("iso", 0.0), **kw)
    assert np.all(reference_correction(so, iso, phi, K, nq, rows) == 0)


@pytest.mark.parametrize("aer,factor", [(("hg", 0.85), 20.0), (("fwc", 0.5), 20.0)])
def test_correction_converges_faster_in_K(so, aer, factor):
    """NumPy restatement of solve_azimuthal (every mode for exactly the orders of mode 0): with the exact single scattering
    the K = 8 radiance is much closer to the K = 48 one than the truncated series are (measured on this grid: 129x for HG
    0.85, 36x for FWC)."""
    sc = small(aer_phase=aer, mu0=0.6)
    mu, nq, K = sos.mu_grid(M_SMALL), 97, 48
    osc = oracle_scenario(so, sc)
    P0a0, Pa0 = sos.phase_matrices("rayleigh", M_SMALL, mu, sc.mu0)
    P0e0, Pe0 = sos.phase_matrices(aer[0], M_SMALL, mu, sc.mu0, aer[1])
    n0 = so.solve(osc, P0a0, Pa0, P0e0, Pe0, method="recurrence", keep_orders=False, use_gemm=True)["n"]
    P0a, Pa = sos.phase_modes("rayleigh", M_SMALL, mu, K, mu0=sc.mu0, n_quad=nq)
    P0e, Pe = sos.phase_modes(aer[0], M_SMALL, mu, K, aer[1], mu0=sc.mu0, n_quad=nq)
    P0a[0], Pa[0], P0e[0], Pe[0] = P0a0, Pa0, P0e0, Pe0   # mode 0 is the base solve
    P0a[3:], Pa[3:] = 0.0, 0.0                           # Rayleigh modes m >= 3 vanish
    rows = [0, 60, L_SMALL - 1]
    modes = np.stack([oracle_mode(so, sc, P0a[m], Pa[m], P0e[m], Pe[m], n0)[rows] for m in range(K)])
    phi = np.concatenate([np.linspace(0, np.pi, 13), [0.05]])

    def series(k):
        w = np.cos(np.arange(k)[:, None] * phi[None, :]) * np.where(np.arange(k) == 0, 1.0, 2.0)[:, None]
        return np.einsum("krn,kp->rpn", modes[:k], w)

    s8, s48 = series(8), series(48)
    c8, c48 = s8 + reference_correction(so, sc, phi, 8, nq, rows), s48 + reference_correction(so, sc, phi, 48, nq, rows)
    assert np.abs(s8 - s48).max() >= factor * np.abs(c8 - c48).max()


def test_bogus_single_scatter_is_refused_before_any_device_work(monkeypatch):
    def no_device(*a, **k):
        raise AssertionError("device work before the ValueError")
    monkeypatch.setattr(AZ, "solved_batches", no_device)
    monkeypatch.setattr(AZ, "BatchSolver", no_device)
    with pytest.raises(ValueError, match="single_scatter"):
        sos.solve_azimuthal([small()], [0.0, np.pi], 4, single_scatter="bogus")


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    sos._lib.load()
    return torch


@pytest.mark.gpu
@pytest.mark.parametrize("aer", [("hg", 0.7), ("fwc", 0.5), ("eva", None)])
def test_first_order_is_exact(gpu, so, aer):
    """max_orders = 1: the corrected radiance is the closed-form first order of P0 = p(cos Theta) / T, whatever K."""
    K, nq, mu0 = 4, 25, 0.5
    sc = small(mu0=mu0, aer_phase=aer, max_orders=1)
    mu = sos.mu_grid(M_SMALL)
    assert np.min(np.abs(mu + mu0)) < 1e-12 and np.min(np.abs(mu - mu0)) < 1e-12   # the |mu -+ mu0| < 1e-4 columns
    phi = np.array([0.0, 0.02, np.pi])
    rows = tuple(range(L_SMALL))
    a = sos.solve_azimuthal([sc], phi, K, rows=rows, n_quad=nq, single_scatter="exact")[0]
    assert a.base.n == 1 and a.single_scatter == "exact"
    osc = oracle_scenario(so, sc)
    tau, _, iu, idn = osc.geometry()
    for p in range(phi.size):
        ex = [PH.phase_exact(s[0], M_SMALL, mu, mu0, phi[p], s[1], nq)[0] for s in (sc.atm_phase, sc.aer_phase)]
        want = so.first_order_regions(osc, tau, mu, iu, idn, *ex)
        assert relmax(a.radiance[:, p], want) <= 1e-12, p


GROUNDS = [dict(surface="specular", grd_alb=0.0), dict(surface="specular", grd_alb=0.3),
           dict(surface="lambert_diffuse", grd_alb=0.3), dict(surface="rossli", grd_alb=0.1, brdf_vol=0.05, brdf_geo=0.02),
           dict(surface="ocean", grd_alb=0.02, wind_speed=5.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("ground", GROUNDS, ids=["black", "specular", "lambert_diffuse", "rossli", "ocean"])
def test_device_correction_matches_the_reference(gpu, so, ground):
    """exact - series is the NumPy reference correction, for a batch that mixes families and mu0 (over the ocean too: the
    glint correction is in both and cancels), at TOA, the surface, inside the aerosol layer and on the region boundaries."""
    scs = [small(mu0=0.5, aer_phase=("hg", 0.8), **ground), small(mu0=0.72, aer_phase=("fwc", 0.5), **ground),
           small(mu0=0.35, atm_phase=("hg", 0.6), aer_phase=("eva", None), **ground),
           small(mu0=0.6, atm_phase=("iso", 0.0), aer_phase=("hg", 0.9), **ground)]
    _, _, iu, idn = oracle_scenario(so, scs[0]).geometry()
    rows = (0, iu - 1, iu, (iu + idn) // 2, idn, idn + 1, L_SMALL - 1)
    phi = np.array([0.0, 0.01, 1.0, np.pi / 2, np.pi, 4.0])
    K, nq = 6, 25
    ser = sos.solve_azimuthal(scs, phi, K, rows=rows, n_quad=nq)
    ex = sos.solve_azimuthal(scs, phi, K, rows=rows, n_quad=nq, single_scatter="exact")
    for a, b, sc in zip(ser, ex, scs):
        want = reference_correction(so, sc, phi, K, nq, rows)
        assert np.abs(want).max() > 1e-3 * np.abs(b.radiance).max()
        assert relmax(b.radiance - a.radiance, want) <= 1e-12, sc


@pytest.mark.gpu
def test_series_is_unchanged(gpu):
    scs = [small(aer_phase=("hg", 0.8)), small(mu0=0.7, aer_phase=("fwc", 0.5))]
    phi = np.linspace(0, np.pi, 5)
    plain = sos.solve_azimuthal(scs, phi, 5)
    ser = sos.solve_azimuthal(scs, phi, 5, single_scatter="series")
    ex = sos.solve_azimuthal(scs, phi, 5, single_scatter="exact")
    for a, b, c in zip(plain, ser, ex):
        assert a.single_scatter == b.single_scatter == "series" and c.single_scatter == "exact"
        assert np.array_equal(a.radiance, b.radiance)
        assert not np.array_equal(a.radiance, c.radiance)
        assert np.array_equal(a.base.I, c.base.I) and np.array_equal(a.modes, c.modes)
        assert np.array_equal(a.mode_orders, c.mode_orders)


@pytest.mark.gpu
@pytest.mark.parametrize("atm,aer", [(("rayleigh", 0.5), ("rayleigh", 0.5)), (("iso", 0.0), ("iso", 0.0)),
                                     (("iso", 0.0), ("rayleigh", 0.5))])
def test_rayleigh_and_isotropic_media_need_no_correction(gpu, atm, aer):
    sc = small(atm_phase=atm, aer_phase=aer)
    phi = np.linspace(0, 2 * np.pi, 9)
    a = sos.solve_azimuthal([sc], phi, 5)[0]
    b = sos.solve_azimuthal([sc], phi, 5, single_scatter="exact")[0]
    assert np.abs(b.radiance - a.radiance).max() <= 1e-13 * np.abs(a.radiance).max()
