"""surface="lambert_diffuse": a Lambertian ground in every order, the direct beam included.

Order 1 is the black-ground closed form (no mirror-reflected beam) plus, on every upward column, the isotropic surface
radiance b_s = rho (e^{-T/mu0} + l(I_1[L-1])) carried up, where l(row) = -2 trapz(row[:M] mu, mu) over the whole downward
half (the lambert_readme trapezoid): the Lambert reflection of the direct beam (irradiance pi e^{-T/mu0} with F0 = pi/mu0)
and of order 1's own downward light.  Orders n >= 2 use the lambert_readme coupling.  The fluxes carry no collimated
reflected beam.

The oracle has no such surface; `diffuse_solve` below restates it from the oracle's own pieces (first_order_regions over a
black ground, order_sweeps with the lambert_readme coupling).  The restatement is checked against the adding identity of a
Lambert boundary, I_rho = I_0 + rho E_rho U with E_rho = E_0 / (1 - rho s), which holds exactly for a linear boundary and
fails if order 1 omits or double-counts the reflected beam or its diffuse part, or reflects it like a mirror.  The oracle's
mu -> 0+ blend (a find-first rule, not linear in rho) is switched off for that identity; the GPU is tied to the oracle with
the blend on.
"""
import dataclasses
from importlib import import_module

import numpy as np
import pytest

from conftest import relelem, relmax

import sos_b200 as sos

AZ = import_module("sos-radiative-transfer_b200.azimuth")

TOL = 1e-10
IDENTITY_KW = dict(nb_layers=60, nb_angles=41, mu0=0.6, tauStar_atm=0.3, tauStar_aer=0.4, alb_aer=0.95, alb_atm=1.0)


@pytest.fixture(scope="module")
def so():
    import sos_oracle
    return sos_oracle


def no_blend(monkeypatch, so):
    monkeypatch.setattr(so, "_blend_row", lambda row, mu, M: M + 1)


def oracle_scenario(so, sc, **kw):
    """The oracle's Scenario with the fields of a drivers Scenario (or keyword arguments)."""
    if sc is not None:
        kw = dict({f.name: getattr(sc, f.name) for f in dataclasses.fields(so.Scenario)}, **kw)
    return so.Scenario(**kw)


def diffuse_first_order(so, osc, tau, mu, iu, idn, P0a, P0e):
    """Order 1 over a diffuse Lambert ground and its surface radiance b_s."""
    M, L = osc.nb_angles, osc.nb_layers
    I1 = so.first_order_regions(dataclasses.replace(osc, grd_alb=0.0, surface="specular"), tau, mu, iu, idn, P0a, P0e)
    T = osc.tauStar_atm + osc.tauStar_aer
    b = osc.grd_alb * (np.exp(-T / osc.mu0) - 2 * so.trapz(I1[L - 1, :M] * mu[:M], mu[:M]))
    up = np.arange(M + 1, 2 * M)
    I1[:, up] += b * np.exp(-(tau[L - 1] - tau)[:, None] / mu[up][None, :])
    return I1, b


def diffuse_solve(so, osc, P0a, Pa, P0e, Pe, keep_orders=False):
    """so.solve(..., method="recurrence", use_gemm=True) with the diffuse Lambert ground; the same loop and stopping rule."""
    tau, z, iu, idn = osc.geometry()
    M, L = osc.nb_angles, osc.nb_layers
    mu = so.mu_grid(M)
    I1, b = diffuse_first_order(so, osc, tau, mu, iu, idn, P0a, P0e)
    lay = so.driver_layout(osc, tau, mu, iu, idn)
    lay.surface = "lambert_readme"
    dtau_aer = osc.tauStar_aer / (idn + 1 - iu)
    dtau_atm = osc.tauStar_atm / L
    f_atm, f_aer = dtau_atm / (dtau_atm + dtau_aer), dtau_aer / (dtau_atm + dtau_aer)
    A_atm = so.contraction_matrix(Pa, mu, osc.alb_atm)
    A_mix = f_atm * A_atm + f_aer * so.contraction_matrix(Pe, mu, osc.alb_aer)
    In_1, I, In, n, saved = I1, I1.copy(), np.ones_like(I1), 1, [I1]
    while True:
        r = so.convergence_ratio(In, I, M)
        if not (r >= osc.threshold) or n >= osc.max_orders:
            break
        n += 1
        J = In_1 @ A_atm
        J[iu: idn + 1] = In_1[iu: idn + 1] @ A_mix
        In = so.order_sweeps(lay, J, method="recurrence")
        In_1 = In
        I = I + In
        if keep_orders:
            saved.append(In)
    return dict(I=I, I_saved=saved, n=n, tau=tau, mu=mu, z=z, idx_up=iu, idx_down=idn, b=b)


def identity_phases(M, mu0):
    mu = sos.mu_grid(M)
    P0a, Pa = sos.phase_matrices("rayleigh", M, mu, mu0, 0.0)
    P0e, Pe = sos.phase_matrices("hg", M, mu, mu0, 0.6)
    return mu, (P0a, Pa, P0e, Pe)


def ground_irradiance(so, I, mu, M, T, mu0):
    """Downward irradiance at the ground over pi: direct e^{-T/mu0} plus diffuse -2 trapz(I[L-1, :M] mu)."""
    return np.exp(-T / mu0) - 2 * so.trapz(I[-1, :M] * mu[:M], mu[:M])


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_adding_identity_on_the_oracle(so, monkeypatch):
    """I_rho = I_0 + rho E_rho U with E_rho = E_0 / (1 - rho s): one spherical albedo s from every rho, and one response U."""
    no_blend(monkeypatch, so)
    M = IDENTITY_KW["nb_angles"]
    T = IDENTITY_KW["tauStar_atm"] + IDENTITY_KW["tauStar_aer"]
    mu, ph = identity_phases(M, IDENTITY_KW["mu0"])
    I, E = {}, {}
    for rho in (0.0, 0.2, 0.5, 0.8):
        ref = diffuse_solve(so, oracle_scenario(so, None, surface="lambert_diffuse", grd_alb=rho, threshold=1e-12,
                                                **IDENTITY_KW), *ph)
        I[rho], E[rho] = ref["I"], ground_irradiance(so, ref["I"], mu, M, T, IDENTITY_KW["mu0"])
    s = {rho: (1 - E[0.0] / E[rho]) / rho for rho in (0.2, 0.5, 0.8)}
    assert 0 < s[0.5] < 1
    assert max(abs(s[r] - s[0.5]) for r in s) <= 1e-9, s
    U = {rho: (I[rho] - I[0.0]) * (1 - rho * s[0.5]) / rho for rho in s}
    err = max(np.abs(U[r] - U[0.5]).max() for r in s) / np.abs(U[0.5]).max()
    assert err <= 1e-10, err


def test_oracle_per_order_invariants(so, monkeypatch):
    """Order 1's upward surface row is b_s on every column >= M+1; order n >= 2's seed is 2 rho down_n (F_up = rho F_down)."""
    no_blend(monkeypatch, so)
    rho = 0.4
    M, L = IDENTITY_KW["nb_angles"], IDENTITY_KW["nb_layers"]
    T = IDENTITY_KW["tauStar_atm"] + IDENTITY_KW["tauStar_aer"]
    mu, ph = identity_phases(M, IDENTITY_KW["mu0"])
    ref = diffuse_solve(so, oracle_scenario(so, None, surface="lambert_diffuse", grd_alb=rho, **IDENTITY_KW), *ph, keep_orders=True)
    I1 = ref["I_saved"][0]
    b = rho * (np.exp(-T / IDENTITY_KW["mu0"]) - 2 * so.trapz(I1[L - 1, :M] * mu[:M], mu[:M]))
    assert b > 0 and np.all(I1[L - 1, M + 1:] == b)
    assert ref["n"] > 3
    for In in ref["I_saved"][1:]:
        down = -so.trapz(In[L - 1, :M] * mu[:M], mu[:M])
        seed = In[L - 1, M + 1:]
        assert down > 0 and np.all(seed == seed[0])
        assert abs(seed[0] - 2 * rho * down) <= 1e-14 * seed[0]


def test_oracle_at_zero_albedo_is_the_black_ground(so):
    M = IDENTITY_KW["nb_angles"]
    _, ph = identity_phases(M, IDENTITY_KW["mu0"])
    d = diffuse_solve(so, oracle_scenario(so, None, surface="lambert_diffuse", grd_alb=0.0, **IDENTITY_KW), *ph)
    s = so.solve(oracle_scenario(so, None, surface="specular", grd_alb=0.0, **IDENTITY_KW), *ph, method="recurrence",
                 use_gemm=True, keep_orders=False)
    assert d["n"] == s["n"] and np.array_equal(d["I"], s["I"])


def test_solve_azimuthal_accepts_the_diffuse_ground(monkeypatch):
    class Reached(Exception):
        pass

    def sentinel(*a, **k):
        raise Reached
    monkeypatch.setattr(AZ, "solved_batches", sentinel)
    sc = sos.Scenario(nb_layers=120, nb_angles=41, surface="lambert_diffuse", grd_alb=0.3)
    with pytest.raises(Reached):
        sos.solve_azimuthal([sc], [0.0, np.pi], 3)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    sos._lib.load()
    return torch


def oracle_for(so, sc, keep_orders=False):
    M = sc.nb_angles
    mu = so.mu_grid(M)
    P0a, Pa = sos.phase_matrices(sc.atm_phase[0], M, mu, sc.mu0, sc.atm_phase[1])
    P0e, Pe = sos.phase_matrices(sc.aer_phase[0], M, mu, sc.mu0, sc.aer_phase[1])
    return diffuse_solve(so, oracle_scenario(so, sc), P0a, Pa, P0e, Pe, keep_orders=keep_orders), mu


def assert_quadratures_match(so, sc, got, ref, mu):
    """Fluxes, diffusivity, heating rate and TOA net flux against the oracle's quadratures without a reflected beam."""
    M, F0 = sc.nb_angles, np.pi / sc.mu0
    up, down = so.flux_up_down(ref["I"], mu, M, ref["tau"], sc.mu0, F0, 0.0)
    assert relmax(got.flux_up, up) < TOL and relmax(got.flux_down, down) < TOL
    assert relmax(got.net_flux, so.net_flux(ref["I"], mu, ref["tau"], sc.mu0, F0, 0.0)) < TOL
    assert relmax(got.diffusivity, so.diffusivity(ref["I"], mu)) < TOL
    hr = so.heating_rate(ref["I"], mu, ref["z"], M, ref["idx_up"], ref["idx_down"], F0, sc.mu0, ref["tau"], 0.0)
    scale = np.max(np.abs(down)) / abs(ref["z"][1] - ref["z"][0]) / (1.225 * 1004)
    assert np.max(np.abs(got.heating_rate - hr)) < TOL * scale
    toa = so.toa_net_flux(ref["I"], mu, M, ref["tau"], sc.mu0, F0, 0.0)
    assert abs(got.toa_net_flux - toa) < TOL * abs(toa)


def mixed_batch(surface="lambert_diffuse", **over):
    base = dict(nb_layers=96, nb_angles=251, atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.5), surface=surface)
    base.update(over)
    return [sos.Scenario(mu0=0.5, tauStar_atm=0.124, tauStar_aer=0.0, grd_alb=0.15, **base),
            sos.Scenario(mu0=0.37, tauStar_atm=0.6, tauStar_aer=0.9, alb_aer=0.8, alb_atm=0.9, grd_alb=0.3, **base),
            sos.Scenario(mu0=0.9, tauStar_atm=0.3, tauStar_aer=0.2, alb_aer=1.0, grd_alb=0.0, **base),
            sos.Scenario(mu0=0.2, tauStar_atm=0.05, tauStar_aer=0.01, alb_aer=0.95, grd_alb=1.0, z_up=60.0, z_down=30.0, **base)]


@pytest.mark.gpu
def test_parity_with_the_oracle(gpu, so):
    """A mixed batch (no aerosol, absorbing gas, rho in {0, 0.15, 0.3, 1}, mu0 on and off the grid, two aerosol layouts),
    an optically thick column (extrapolation widths 0.02 M above, 0.06 M below) and drivers-size rows (M = 501)."""
    thick = sos.Scenario(nb_layers=400, nb_angles=151, mu0=0.37, tauStar_atm=0.8, tauStar_aer=3.6, alb_aer=0.8, alb_atm=0.9,
                         grd_alb=0.3, z_up=100.0, z_down=10.0, surface="lambert_diffuse", atm_phase=("rayleigh", 0.0),
                         aer_phase=("hg", 0.5))
    wide = sos.Scenario(nb_layers=120, nb_angles=501, mu0=0.6, tauStar_atm=0.124, tauStar_aer=0.12, alb_aer=0.97, grd_alb=0.15,
                        surface="lambert_diffuse", atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.7))
    scs = mixed_batch() + [thick, wide]
    got = sos.solve_scenarios(scs)
    worst = 0.0
    for i, (sc, r) in enumerate(zip(scs, got)):
        ref, mu = oracle_for(so, sc)
        assert r.n == ref["n"], (i, r.n, ref["n"])
        assert r.status == 0, (i, r.status)
        err = relmax(r.I, ref["I"])
        worst = max(worst, err)
        assert err < TOL and relelem(r.I, ref["I"]) < 1e-8, (i, err)
        assert_quadratures_match(so, sc, r, ref, mu)
    print(f"lambert_diffuse parity: worst relmax {worst:.2e}")


@pytest.mark.gpu
def test_zero_albedo_equals_the_black_specular_ground(gpu):
    scs = [dataclasses.replace(sc, grd_alb=0.0) for sc in mixed_batch()]
    a = sos.solve_scenarios(scs)
    b = sos.solve_scenarios([dataclasses.replace(sc, surface="specular") for sc in scs])
    for x, y in zip(a, b):
        assert x.n == y.n and x.status == y.status and np.array_equal(x.I, y.I)
        for q in ("flux_up", "flux_down", "net_flux", "diffusivity", "heating_rate"):
            assert np.array_equal(getattr(x, q), getattr(y, q)), q
        assert x.toa_net_flux == y.toa_net_flux


@pytest.mark.gpu
def test_per_order_invariants_on_the_device(gpu, so):
    kw = dict(nb_layers=120, nb_angles=101, mu0=0.6, tauStar_atm=0.3, tauStar_aer=0.4, alb_aer=0.95, grd_alb=0.4)
    sc = sos.Scenario(atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.6), surface="lambert_diffuse", **kw)
    r = sos.solve_scenarios([sc], keep_orders=6)[0]
    M, mu, L = sc.nb_angles, r.mu, sc.nb_layers
    T = sc.tauStar_atm + sc.tauStar_aer
    I1 = r.I_saved[0]
    b = sc.grd_alb * (np.exp(-T / sc.mu0) - 2 * so.trapz(I1[L - 1, :M] * mu[:M], mu[:M]))
    row = I1[L - 1, M + 1:]
    assert b > 0
    assert np.max(np.abs(row - row[0])) <= 1e-14 * row[0]          # isotropic
    assert np.max(np.abs(row - b)) <= 1e-14 * b
    for n in range(1, min(6, r.n)):                                  # orders 2 ..
        In = r.I_saved[n]
        down = -so.trapz(In[L - 1, :M] * mu[:M], mu[:M])
        seed = In[L - 1, M + 40:]                                    # away from the mu -> 0+ blend
        assert down > 0 and np.all(seed > 0)
        assert np.max(np.abs(seed - seed[0])) < 1e-13 * abs(seed[0])
        assert abs(seed[0] - 2 * sc.grd_alb * down) < 1e-12 * abs(seed[0])
    # the per-order fields match the oracle's
    ref, _ = oracle_for(so, sc, keep_orders=True)
    assert r.n == ref["n"]
    for n in range(min(6, r.n)):
        assert relmax(r.I_saved[n], ref["I_saved"][n]) < TOL, n


@pytest.mark.gpu
def test_first_order_entry_points_agree_bit_for_bit(gpu):
    """sos_first_order, sos_first_order2 (with its second destination) and sos_first_order_tab write the same bits."""
    torch = gpu
    scen = [sos.Scenario(nb_layers=90, nb_angles=75, tauStar_atm=0.124, tauStar_aer=0.03 + 0.05 * i, mu0=(0.2, 0.5, 0.9)[i % 3],
                         alb_aer=0.8 + 0.02 * i, grd_alb=0.1 * (i % 4), atm_phase=("rayleigh", 0.0),
                         aer_phase=(("hg", 0.5), ("hg", 0.7), ("fwc", 0.0))[i % 3], surface="lambert_diffuse") for i in range(9)]
    bs = sos.BatchSolver(scen)
    eng = bs.engine
    try:
        assert eng.table_fits(bs.P0tab.shape[0], len(scen), eng.N)
        acc = eng.new_field(zero=True)
        a = bs.first_order(also_into=acc).clone()
        b = eng.first_order(bs.Ccoef)
        C = np.ascontiguousarray(bs.Ccoef)
        c = eng.new_field(zero=True)
        sos._lib.check(eng.lib.sos_first_order(eng._plan, C.ctypes.data, c.data_ptr(), eng._stream), "sos_first_order")
        torch.cuda.synchronize()
        assert torch.equal(a, b) and torch.equal(a, c)
        assert torch.equal(acc[:, : eng.N], a[:, : eng.N])
        assert float(a[:, : eng.N].abs().max()) > 0
    finally:
        eng.close()


@pytest.mark.gpu
def test_generated_source_equals_stored_source(gpu, monkeypatch):
    scs = mixed_batch()[:3] + mixed_batch(nb_layers=130, nb_angles=501)[:3]
    outs = {}
    for flag in ("1", "0"):
        monkeypatch.setenv("SOS_B200_GENSRC", flag)
        outs[flag] = sos.solve_scenarios(scs, keep_orders=3)
    for x, y in zip(outs["1"], outs["0"]):
        assert x.n == y.n and x.status == y.status
        assert relmax(x.I, y.I) <= 1e-12
        for p, q in zip(x.I_saved, y.I_saved):
            assert relmax(p, q) <= 1e-12
        assert relmax(x.flux_up, y.flux_up) <= 1e-12 and abs(x.toa_net_flux - y.toa_net_flux) <= 1e-12 * abs(y.toa_net_flux)


@pytest.mark.gpu
def test_plan_reuse_equals_fresh_solvers(gpu):
    """BatchSolver.update over three batches (new tau, mu0, albedos) against a fresh solver per batch, bit for bit: the
    plan's surface-radiance buffer is rewritten by every first order."""
    first = mixed_batch()[:3]
    batches = [first,
               [dataclasses.replace(sc, mu0=0.3 + 0.2 * i, grd_alb=0.6 - 0.1 * i, tauStar_atm=0.2 + 0.1 * i)
                for i, sc in enumerate(first)],
               [dataclasses.replace(sc, grd_alb=1.0, alb_aer=0.9, tauStar_aer=0.05 * (i + 1)) for i, sc in enumerate(first)]]
    reused = sos.BatchSolver(batches[0])
    try:
        for k, batch in enumerate(batches):
            if k:
                reused.update(batch)
            got = reused.results(reused.solve(), quadratures=True)
            fresh = sos.BatchSolver(batch)
            try:
                want = fresh.results(fresh.solve(), quadratures=True)
            finally:
                fresh.engine.close()
            for x, y in zip(got, want):
                assert x.n == y.n and x.status == y.status and np.array_equal(x.I, y.I), k
                assert np.array_equal(x.flux_up, y.flux_up) and x.toa_net_flux == y.toa_net_flux, k
    finally:
        reused.engine.close()


@pytest.mark.gpu
def test_critical_albedo_sweep_forcing_is_the_toa_difference(gpu):
    base = dict(nb_layers=96, nb_angles=101, atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.7), surface="lambert_diffuse")
    pts = [sos.Scenario(mu0=0.5, tauStar_atm=0.124, tauStar_aer=0.12, grd_alb=0.15, **base),
           sos.Scenario(mu0=0.7, tauStar_atm=0.124, tauStar_aer=0.3, grd_alb=0.6, **base),
           sos.Scenario(mu0=0.3, tauStar_atm=0.2, tauStar_aer=0.05, grd_alb=0.3, **base)]
    omega_c, forcing, n_solves, omega = sos.critical_albedo_sweep(pts, return_evaluated=True)
    assert n_solves > len(pts) and np.all(np.isfinite(forcing))
    for p, w, f in zip(pts, omega, forcing):
        with_aer = sos.solve_scenarios([dataclasses.replace(p, alb_aer=float(w))])[0].toa_net_flux
        without = sos.solve_scenarios([dataclasses.replace(p, tauStar_aer=0.0, alb_aer=1.0)])[0].toa_net_flux
        assert abs(f - (with_aer - without)) <= 1e-10 * max(abs(with_aer), abs(without))


@pytest.mark.gpu
def test_azimuth_over_the_diffuse_ground(gpu, so):
    """Mode 0 carries the ground (base = solve_scenarios bit for bit); modes 1 and 2 are those of a black ground summed for
    exactly n_0 orders; the azimuth mean of the synthesized radiance is mode 0."""
    from test_azimuth import L_SMALL, M_SMALL, oracle_mode
    K = 5
    scs = [sos.Scenario(nb_layers=L_SMALL, nb_angles=M_SMALL, mu0=mu0, tauStar_atm=0.124, tauStar_aer=0.12, grd_alb=rho,
                        alb_aer=0.97, atm_phase=("rayleigh", 0.5), aer_phase=("hg", g), surface="lambert_diffuse")
           for mu0, rho, g in ((0.5, 0.3, 0.5), (0.8, 0.15, 0.7))]
    phi = np.arange(2 * K + 3) * (2 * np.pi / (2 * K + 3))
    az = sos.solve_azimuthal(scs, phi, K, rows=tuple(range(L_SMALL)), n_quad=25)
    ref = sos.solve_scenarios(scs)
    for a, r, sc in zip(az, ref, scs):
        assert np.array_equal(a.base.I, r.I) and a.base.n == r.n and a.base.toa_net_flux == r.toa_net_flux
        n0 = r.n
        assert np.all(a.mode_orders == n0) and np.all(a.mode_status == 0), (a.mode_orders, a.mode_status)
        mu = sos.mu_grid(M_SMALL)
        P0a, Pa = sos.phase_modes("rayleigh", M_SMALL, mu, K, mu0=sc.mu0)
        P0e, Pe = sos.phase_modes("hg", M_SMALL, mu, K, sc.aer_phase[1], mu0=sc.mu0)
        black = dataclasses.replace(sc, surface="specular", grd_alb=0.0)
        for m in (1, 2):
            want = oracle_mode(so, black, P0a[m], Pa[m], P0e[m], Pe[m], n0)
            assert relmax(a.modes[m], want) <= TOL and relelem(a.modes[m], want) <= TOL, m
        assert relmax(a.radiance.mean(axis=1), a.base.I[a.rows]) <= 1e-13


@pytest.mark.gpu
def test_single_layer_plan_refuses_the_diffuse_ground(gpu):
    """The diffuse ground needs the three-region first order: a single-layer plan answers SOS_ERR_UNSUPPORTED."""
    E = import_module("sos-radiative-transfer_b200.engine")
    M, L = 41, 32
    mu = sos.mu_grid(M)
    tau = np.linspace(0.0, 0.5, L)
    w = sos.grid.extrapolation_width(float(tau[-1]), M)
    sc = E.ScenarioCoefficients(mu0=0.5, grd_alb=0.3, tauStar_tot=0.5, coef_atm=1.0, extrap_width=(w, w, w))
    with pytest.raises(sos._lib.SosError, match=r"\(-4\)"):
        E.SosEngine(mu, tau[None, :], [sc], region_start=[0, L], surface=sos._lib.SURFACE_LAMBERT_DIFFUSE)
