"""Azimuth-resolved radiance: Fourier modes of the phase functions (phase.phase_modes, sos_build_phase_modes), mode members
with an order cap, device synthesis (sos_azimuth_synthesis) and solve_azimuthal.

phi is the azimuth of the propagation direction of the diffuse light relative to that of the solar beam (the beam travels
along (-mu0, 0): cos Theta = -mu0 mu + sqrt(1 - mu0^2) sqrt(1 - mu^2) cos phi, phi = 0 forward).
"""
import dataclasses
from importlib import import_module

import numpy as np
import pytest

from conftest import relelem, relmax

import sos_b200 as sos

PH = import_module("sos-radiative-transfer_b200.phase")
AZ = import_module("sos-radiative-transfer_b200.azimuth")

M_SMALL, L_SMALL = 41, 120
FAMILIES = [("rayleigh", 0.5), ("hg", 0.7), ("fwc", 0.5), ("mie_lognormal", sos.EVA_AEROSOL)]


def hg(g):
    return lambda c: (1 - g * g) / (1 + g * g - 2 * g * c) ** 1.5


def cos_theta(mu, mu0, phi):
    return -mu0 * mu[:, None] + np.sqrt(1 - mu0 ** 2) * np.sqrt(1 - mu ** 2)[:, None] * np.cos(phi)[None, :]


def synthesize(P0m, phi):
    K = P0m.shape[0]
    return P0m[0][:, None] + 2 * np.einsum("kn,kp->np", P0m[1:], np.cos(np.arange(1, K)[:, None] * phi[None, :]))


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name,g", FAMILIES)
def test_mode_zero_is_the_azimuth_average(name, g):
    mu = sos.mu_grid(M_SMALL)
    P0m, Pm = sos.phase_modes(name, M_SMALL, mu, 4, g, mu0=0.6)
    assert P0m.shape == (4, 2 * M_SMALL) and Pm.shape == (4, 2 * M_SMALL, 2 * M_SMALL)
    assert np.array_equal(P0m[0], sos.phase_P0(name, M_SMALL, mu, 0.6, g))
    assert np.array_equal(Pm[0], sos.phase_P(name, M_SMALL, mu, g))


def test_rayleigh_modes_closed_forms():
    mu = sos.mu_grid(M_SMALL)
    P0m, Pm = sos.phase_modes("rayleigh", M_SMALL, mu, 6, mu0=0.6)
    top = np.abs(Pm).max()
    assert np.abs(Pm[3:]).max() < 1e-15 * top and np.abs(P0m[3:]).max() < 1e-15 * np.abs(P0m).max()
    s = np.sqrt(1 - mu * mu)
    # 0.75 (1 + cos^2 Theta): mode 1 ~ mu mu' s s', mode 2 ~ s^2 s'^2 (columns scaled by the mode-0 normalisation)
    for m, shape in ((1, np.outer(mu * s, mu * s)), (2, np.outer(s * s, s * s))):
        ratio = Pm[m][shape != 0] / shape[shape != 0]
        col = np.broadcast_to(np.arange(2 * M_SMALL)[None, :], shape.shape)[shape != 0]
        for n in np.unique(col)[::7]:
            r = ratio[col == n]
            assert np.ptp(r) <= 1e-12 * np.abs(r).max()
        assert np.abs(Pm[m][shape == 0]).max() < 1e-15 * top


def test_isotropic_modes_vanish():
    mu = sos.mu_grid(M_SMALL)
    P0m, Pm = sos.phase_modes("iso", M_SMALL, mu, 5, mu0=0.5)
    assert np.all(P0m[1:] == 0) and np.all(Pm[1:] == 0)
    assert np.all(P0m[0] == 1) and np.all(Pm[0] == 2)


@pytest.mark.parametrize("name,g", FAMILIES[:3])
def test_every_mode_is_centrosymmetric(name, g):
    """P_m(mu, mu') = P_m(-mu, -mu'): the precondition of the folded contraction."""
    mu = sos.mu_grid(M_SMALL)
    _, Pm = sos.phase_modes(name, M_SMALL, mu, 6, g, n_quad=49)
    for m in range(6):
        assert np.abs(Pm[m] - Pm[m][::-1, ::-1]).max() <= 1e-13 * np.abs(Pm).max()


@pytest.mark.parametrize("name,f,K,n_quad,tol", [("rayleigh", lambda c: 0.75 * (1 + c * c), 3, 25, 1e-12),
                                                  ("hg", hg(0.5), 64, 361, 1e-8)])
def test_synthesis_identity(name, f, K, n_quad, tol):
    """sum_m (2 - delta_m0) P0_m cos(m phi) = c p(cos Theta(mu, mu0, phi)) with one constant c."""
    mu, mu0 = sos.mu_grid(M_SMALL), 0.6
    P0m, _ = sos.phase_modes(name, M_SMALL, mu, K, 0.5, mu0=mu0, n_quad=n_quad, want_P=False)
    phi = np.linspace(0, 2 * np.pi, 37)
    c = synthesize(P0m, phi) / f(cos_theta(mu, mu0, phi))
    assert np.abs(c / c.mean() - 1).max() <= tol


@pytest.mark.parametrize("bad", [dict(surface="lambert", grd_alb=0.3), dict(surface="lambert_readme", grd_alb=0.1),
                                 dict(aer_phase=(np.ones(82), 2 * np.ones((82, 82)))), dict(n_quad=9)])
def test_refused_before_any_device_work(bad, monkeypatch):
    kw = dict(bad)
    n_quad = kw.pop("n_quad", 25)
    sc = sos.Scenario(nb_layers=L_SMALL, nb_angles=M_SMALL, **kw)

    def no_device(*a, **k):
        raise AssertionError("device work before the ValueError")
    monkeypatch.setattr(AZ, "solved_batches", no_device)
    monkeypatch.setattr(AZ, "BatchSolver", no_device)
    with pytest.raises(ValueError):
        sos.solve_azimuthal([sc], [0.0, np.pi], 5, n_quad=n_quad)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    sos._lib.load()
    return torch


@pytest.fixture(scope="module")
def so():
    import sos_oracle
    return sos_oracle


def small(**kw):
    base = dict(nb_layers=L_SMALL, nb_angles=M_SMALL, tauStar_atm=0.124, tauStar_aer=0.12, grd_alb=0.3, alb_aer=0.97,
                atm_phase=("rayleigh", 0.5), aer_phase=("hg", 0.5), surface="specular")
    base.update(kw)
    return sos.Scenario(**base)


def oracle_mode(so, sc, P0a, Pa, P0e, Pe, n):
    """The oracle's three-region order loop on one mode's operands for exactly n orders (no ratio test)."""
    osc = so.Scenario(**{f.name: getattr(sc, f.name) for f in dataclasses.fields(so.Scenario)})
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


@pytest.mark.gpu
@pytest.mark.parametrize("name,g", FAMILIES[:3])
def test_device_mode_builder(gpu, name, g):
    bs = sos.BatchSolver([small()])
    eng = bs.engine
    try:
        mu = eng.mu
        P, P0 = eng.build_phase_matrix(name, g, mu0=0.6)
        Pm, P0m = eng.build_phase_modes(name, g, n_modes=6, mu0=0.6, n_quad=25)
        assert gpu.equal(Pm[0], P) and gpu.equal(P0m[0], P0)
        hP0, hP = sos.phase_modes(name, M_SMALL, mu, 6, g, mu0=0.6, n_quad=25)
        assert np.abs(Pm.cpu().numpy()[1:] - hP[1:]).max() <= 1e-12 * np.abs(hP[0]).max()
        assert np.abs(P0m.cpu().numpy()[1:] - hP0[1:]).max() <= 1e-12 * np.abs(hP0[0]).max()
        # more nodes and modes than the azimuth-averaged builders have
        Pm, P0m = eng.build_phase_modes(name, g, n_modes=40, mu0=0.3, n_quad=1024)
        hP0, hP = sos.phase_modes(name, M_SMALL, mu, 40, g, mu0=0.3, n_quad=1024)
        assert np.abs(Pm.cpu().numpy() - hP).max() <= 1e-12 * np.abs(hP[0]).max()
        assert np.abs(P0m.cpu().numpy() - hP0).max() <= 1e-12 * np.abs(hP0[0]).max()
    finally:
        eng.close()


@pytest.mark.gpu
def test_base_is_solve_scenarios_and_modes_match_the_oracle(gpu, so):
    scs = [small(mu0=0.5), small(mu0=0.8, aer_phase=("hg", 0.7))]
    K = 6
    az = sos.solve_azimuthal(scs, np.linspace(0, np.pi, 7), K, rows=tuple(range(L_SMALL)), n_quad=25)
    ref = sos.solve_scenarios(scs)
    for a, r, sc in zip(az, ref, scs):
        assert np.array_equal(a.base.I, r.I) and a.base.n == r.n
        for q in ("flux_up", "flux_down", "net_flux", "diffusivity", "heating_rate"):
            assert np.array_equal(getattr(a.base, q), getattr(r, q)), q
        n0 = r.n
        assert np.all(a.mode_orders == n0) and np.all(a.mode_status == 0), (a.mode_orders, a.mode_status)
        mu = sos.mu_grid(M_SMALL)
        P0a, Pa = sos.phase_modes("rayleigh", M_SMALL, mu, K, mu0=sc.mu0)
        P0e, Pe = sos.phase_modes("hg", M_SMALL, mu, K, sc.aer_phase[1], mu0=sc.mu0)
        for m in (1, 2, 5):
            want = oracle_mode(so, sc, P0a[m], Pa[m], P0e[m], Pe[m], n0)
            assert relmax(a.modes[m], want) <= 1e-10 and relelem(a.modes[m], want) <= 1e-10, m
        # the synthesized radiance is I_0 + 2 sum I_m cos(m phi) of those modes
        syn = a.modes[0][:, None, :] + 2 * np.einsum("krn,kp->rpn", a.modes[1:], np.cos(np.arange(1, K)[:, None] * a.phi[None, :]))
        assert relmax(a.radiance, syn) <= 1e-13


@pytest.mark.gpu
def test_default_grid(gpu):
    scs = [sos.Scenario(**sos.EVA, aer_phase=("hg", 0.7))]
    az = sos.solve_azimuthal(scs, np.linspace(0, np.pi, 5), 4, n_quad=25)
    r = sos.solve_scenarios(scs)[0]
    a = az[0]
    assert np.array_equal(a.base.I, r.I) and a.base.n == r.n
    assert np.all(a.mode_orders == r.n) and np.all(a.mode_status == 0)
    assert a.radiance.shape == (2, 5, 1002) and np.all(np.isfinite(a.radiance))


@pytest.mark.gpu
def test_isotropic_medium_has_no_azimuth_dependence(gpu):
    sc = small(atm_phase=("iso", 0.0), aer_phase=("iso", 0.0))
    a = sos.solve_azimuthal([sc], np.linspace(0, 2 * np.pi, 9), 5)[0]
    rows = a.base.I[a.rows]
    assert np.array_equal(a.radiance, np.broadcast_to(rows[:, None, :], a.radiance.shape))
    assert np.all(a.mode_orders[1:] == 0)


@pytest.mark.gpu
def test_rayleigh_needs_three_modes(gpu):
    sc = small(aer_phase=("rayleigh", 0.5))
    phi = np.linspace(0, 2 * np.pi, 13)
    a3 = sos.solve_azimuthal([sc], phi, 3)[0]
    a8 = sos.solve_azimuthal([sc], phi, 8)[0]
    assert relmax(a8.radiance, a3.radiance) <= 1e-13


@pytest.mark.gpu
def test_azimuth_mean_is_mode_zero(gpu):
    K = 6
    phi = np.arange(2 * K + 3) * (2 * np.pi / (2 * K + 3))
    sc = small(aer_phase=("hg", 0.6))
    a = sos.solve_azimuthal([sc], phi, K)[0]
    assert relmax(a.radiance.mean(axis=1), a.base.I[a.rows]) <= 1e-13


@pytest.mark.gpu
def test_convention_first_order_forward_peak(gpu, so):
    """max_orders = 1: the synthesized first order is the first order of the direct P0(mu; phi) = c p(cos Theta)."""
    g, mu0, K, nq = 0.7, 0.5, 64, 361
    sc = small(mu0=mu0, grd_alb=0.0, atm_phase=("hg", g), aer_phase=("hg", g), max_orders=1)
    phi = np.array([0.0, np.pi / 3, np.pi / 2, np.pi])
    a = sos.solve_azimuthal([sc], np.linspace(0, 2 * np.pi, 73), K, rows=(-1, L_SMALL // 2), n_quad=nq)[0]
    at = sos.solve_azimuthal([sc], phi, K, rows=(-1, L_SMALL // 2), n_quad=nq)[0]
    assert a.base.n == 1
    mu = sos.mu_grid(M_SMALL)
    P0m, _ = sos.phase_modes("hg", M_SMALL, mu, K, g, mu0=mu0, n_quad=nq, want_P=False)
    c = float(np.mean(synthesize(P0m, phi) / hg(g)(cos_theta(mu, mu0, phi))))
    P0dir = c * hg(g)(cos_theta(mu, mu0, phi))
    for p in (0, 3):   # phi = 0 and pi
        osc = so.Scenario(**{f.name: getattr(sc, f.name) for f in dataclasses.fields(so.Scenario)})
        tau, _, iu, idn = osc.geometry()
        want = so.first_order_regions(osc, tau, mu, iu, idn, P0dir[:, p], P0dir[:, p])[at.rows]
        assert relmax(at.radiance[:, p, :], want) <= 1e-6, p
    col = int(np.argmin(np.abs(mu + mu0)))
    assert abs(mu[col] + mu0) < 1e-12
    assert int(np.argmax(a.radiance[0, :, col])) in (0, a.phi.size - 1)   # phi = 0 (= 2 pi): the forward direction


@pytest.mark.gpu
def test_two_plans_accumulate(gpu, monkeypatch):
    scs = [small(mu0=0.5), small(mu0=0.7, aer_phase=("hg", 0.8))]
    phi = np.linspace(0, np.pi, 9)
    one = sos.solve_azimuthal(scs, phi, 5)
    monkeypatch.setattr(AZ, "MODE_PHASES_PER_PLAN", 4)   # two modes per plan: several plans instead of one
    split = sos.solve_azimuthal(scs, phi, 5)
    for a, b in zip(one, split):
        assert relmax(b.radiance, a.radiance) <= 1e-13
        assert np.array_equal(a.mode_orders, b.mode_orders)


@pytest.mark.gpu
def test_zero_operand_keeps_the_fold(gpu):
    """An isotropic aerosol's modes m >= 1 are all-zero operands: centrosymmetric (defect 0), the plan stays folded."""
    sc = small(aer_phase=("iso", 0.0))
    m = dataclasses.replace(sc, atm_phase=("rayleigh", 0.5, 1, 25), aer_phase=("iso", 0.0, 1, 25))
    bs = sos.BatchSolver([m], order_caps=[3])
    try:
        assert bs.engine.folded
        res = bs.solve(max_orders=3)
        assert res.n_orders[0] == 3 and res.status[0] == 0
    finally:
        bs.engine.close()
