"""surface="ocean": a wind-roughened sea (Cox-Munk glint) in every order and azimuthal mode.

rho = grd_alb + rho_glint(W, n).  grd_alb is the 'lambert_diffuse' coupling unchanged; the glint is the one-matrix form of
the Ross-Li coupling, so the oracle construction of test_rossli.py serves unchanged: `rossli_solve` with the glint mode
matrix as the first kernel (weight 1) and a zero second kernel.  solve_azimuthal adds the once-reflected direct beam in
closed form (sos_glint_correction), checked here against the reflectance itself over a non-scattering atmosphere.
"""
import dataclasses
from importlib import import_module

import numpy as np
import pytest

from conftest import relelem, relmax
from test_lambert_diffuse import TOL, IDENTITY_KW, assert_quadratures_match, identity_phases, no_blend, oracle_scenario
from test_rossli import down_weights, rossli_solve

import sos_b200 as sos

OC = sos.ocean
AZ = import_module("sos-radiative-transfer_b200.azimuth")
DR = import_module("sos-radiative-transfer_b200.drivers")
E = import_module("sos-radiative-transfer_b200.engine")
ANGLES = (0.2, 0.3, 0.5, 0.8, 0.95)


@pytest.fixture(scope="module")
def so():
    import sos_oracle
    return sos_oracle


def glint_ground(M, mu, mu0, W, n=OC.OCEAN_INDEX, m=0, K=None):
    """(R, 0, beta, 0) of mode m: the glint as the first kernel of the Ross-Li construction, a zero second kernel."""
    K = m + 1 if K is None else K
    R = OC.glint_modes(M, mu, W, n, K)[m]
    b = OC.glint_beam(M, mu, mu0, W, n, K)[m]
    return R, np.zeros_like(R), b, np.zeros_like(b)


def solve_ref(so, sc, gr=None, **kw):
    M = sc.nb_angles
    mu = so.mu_grid(M)
    P0a, Pa = sos.phase_matrices(sc.atm_phase[0], M, mu, sc.mu0, sc.atm_phase[1])
    P0e, Pe = sos.phase_matrices(sc.aer_phase[0], M, mu, sc.mu0, sc.aer_phase[1])
    gr = glint_ground(M, mu, sc.mu0, sc.wind_speed, sc.ocean_index) if gr is None else gr
    return rossli_solve(so, oracle_scenario(so, sc), P0a, Pa, P0e, Pe, 1.0, 0.0, *gr, **kw), mu


def directional_albedo(M, mu, W):
    """sum_c 2 w_c mu_c rho_0(mu_i, mu_c) for every upward column i."""
    return OC.glint_modes(M, mu, W, n_modes=1)[0] @ down_weights(mu, M)


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_closed_form_at_the_specular_geometry():
    """mu_i = mu_v = mu, phi = 0: mu_n = 1 and rho_glint = r(mu) S / (4 sigma^2 mu^2)."""
    mu = np.array(ANGLES + (1.0,))
    for W in (0.0, 1.0, 7.0, 20.0):
        s2 = OC.slope_variance(W)
        S = 1.0 / (1.0 + 2.0 * OC.smith_lambda(mu, np.sqrt(s2)))
        want = OC.fresnel(mu, 1.34) * S / (4.0 * s2 * mu * mu)
        got = OC.cox_munk(mu, mu, 0.0, W)
        assert np.max(np.abs(got - want) / want) <= 1e-14, W
    assert OC.smith_lambda(1.0, 0.1) == 0.0
    assert abs(OC.fresnel(1.0, 1.34) - (0.34 / 2.34) ** 2) <= 1e-16


def test_reciprocity():
    rng = np.random.default_rng(5)
    a, b, phi = rng.uniform(0.01, 1, 300), rng.uniform(0.01, 1, 300), rng.uniform(0, np.pi, 300)
    for W in (0.0, 3.0, 12.0):
        assert np.array_equal(OC.cox_munk(a, b, phi, W), OC.cox_munk(b, a, phi, W))
    M, K = 31, 5
    mu = sos.mu_grid(M)
    R = OC.glint_modes(M, mu, 4.0, 1.33, K)
    assert R.shape == (K, M - 1, M) and np.all(R[:, :, M - 1] == 0)     # the column mu = 0- is 0
    swapped = R[:, :, : M - 1][:, ::-1, ::-1].transpose(0, 2, 1)
    # (|mu[c]| and mu[M+1+(M-2-c)] differ by an ulp on some columns, and the glint is steep at grazing angles)
    assert np.max(np.abs(R[:, :, : M - 1] - swapped)) <= 1e-11 * np.max(np.abs(R))


def test_albedo_on_the_default_grid():
    """Directional albedo in [0, 1) and, at normal incidence, within 1 % of the Fresnel reflectance r(1) up to 15 m/s (1.0 %
    at 30 m/s, where the wider lobe reaches angles with a larger Fresnel reflectance).  A calm sea
    (W = 0) is the exception on the four most grazing columns (mu <= 0.008), whose lobe the M = 501 grid does not resolve
    (their albedo converges to about 0.74 on finer grids); their quadrature weight mu is below 0.008."""
    M = 501
    mu = sos.mu_grid(M)
    up = mu[M + 1:]
    r1 = OC.fresnel(1.0, 1.34)
    for W in (0.0, 1.0, 5.0, 15.0, 30.0):
        alb = directional_albedo(M, mu, W)
        ok = up > 0.01 if W == 0 else np.ones(up.size, dtype=bool)
        assert np.all(alb >= 0) and np.all(alb[ok] < 1), W
        assert abs(alb[-1] - r1) <= (0.01 if W <= 15 else 0.011) * r1, (W, alb[-1], r1)
        if W == 0:
            assert np.all(up[alb >= 1] <= 0.008)


def test_the_glint_is_forward():
    phi = np.linspace(0, np.pi, 361)
    for mu0 in ANGLES:
        for W in (0.0, 2.0, 10.0):
            assert int(np.argmax(OC.cox_munk(mu0, mu0, phi, W))) == 0


def test_synthesis_error_of_64_modes():
    """At W >= 10 m/s, 64 modes reproduce the glint to 1e-5 of its peak on the angle set; at W = 1 they do not."""
    K = 64
    phi = np.linspace(0, np.pi, 361)
    mu = np.array(ANGLES)
    a, b = np.repeat(mu, mu.size), np.tile(mu, mu.size)
    for W, lo, hi in ((10.0, 0.0, 1e-5), (20.0, 0.0, 1e-5), (1.0, 0.05, 1.0)):
        modes = OC._modes(a, b, W, OC.OCEAN_INDEX, K, sos.BRDF_NODES)            # (K, pairs)
        direct = OC.cox_munk(a[None, :], b[None, :], phi[:, None], W)
        err = np.max(np.abs(sos.brdf.brdf_synthesis(modes, phi) - direct)) / np.max(direct)
        assert lo <= err <= hi, (W, err)


def construction(so, W, n=1.34, **kw):
    M = IDENTITY_KW["nb_angles"]
    mu, ph = identity_phases(M, IDENTITY_KW["mu0"])
    osc = oracle_scenario(so, None, surface="ocean", grd_alb=0.0, **IDENTITY_KW)
    return rossli_solve(so, osc, *ph, 1.0, 0.0, *glint_ground(M, mu, IDENTITY_KW["mu0"], W, n), **kw), mu, ph


def test_per_order_seeds_and_order_one(so, monkeypatch):
    """grd_alb = 0: order 1 is the black ground's plus b e^{-(T - tau)/mu} on the upward columns with b = E beta + R u_1;
    order n's upward surface row is R u_n of its own downward half."""
    no_blend(monkeypatch, so)
    W = 3.0
    ref, mu, ph = construction(so, W, keep_orders=True)
    M, L = IDENTITY_KW["nb_angles"], IDENTITY_KW["nb_layers"]
    R, _, beta, _ = glint_ground(M, mu, IDENTITY_KW["mu0"], W)
    osc = oracle_scenario(so, None, surface="specular", grd_alb=0.0, **IDENTITY_KW)
    tau, _, iu, idn = osc.geometry()
    black = so.first_order_regions(osc, tau, mu, iu, idn, ph[0], ph[2])
    I1 = ref["I_saved"][0]
    T = IDENTITY_KW["tauStar_atm"] + IDENTITY_KW["tauStar_aer"]
    b = np.exp(-T / IDENTITY_KW["mu0"]) * beta + R @ (down_weights(mu, M) * black[L - 1, :M])
    assert np.max(np.abs(ref["b"] - b)) <= 1e-15 * np.max(b)
    up = np.arange(M + 1, 2 * M)
    want = black.copy()
    want[:, up] += b[None, :] * np.exp(-(tau[L - 1] - tau)[:, None] / mu[up][None, :])
    assert np.array_equal(I1, want)
    assert ref["n"] > 3 and np.ptp(b) > 0.05 * np.max(b)
    for In in ref["I_saved"][1:]:
        seed = R @ (down_weights(mu, M) * In[L - 1, :M])
        assert np.max(np.abs(In[L - 1, M + 1:] - seed)) <= 1e-14 * np.max(np.abs(seed))


def test_refusals_before_any_device_work():
    kw = dict(nb_layers=60, nb_angles=41)
    bad = [sos.Scenario(surface="ocean", grd_alb=0.02, **kw),
           sos.Scenario(surface="ocean", grd_alb=0.02, wind_speed=-1.0, **kw),
           sos.Scenario(surface="ocean", grd_alb=0.02, wind_speed=float("nan"), **kw),
           sos.Scenario(surface="ocean", grd_alb=0.02, wind_speed=5.0, ocean_index=1.0, **kw),
           sos.Scenario(surface="ocean", grd_alb=0.02, wind_speed=5.0, ocean_index=float("inf"), **kw),
           sos.Scenario(surface="specular", grd_alb=0.1, wind_speed=5.0, **kw),
           sos.Scenario(surface="rossli", grd_alb=0.1, brdf_vol=0.1, wind_speed=5.0, **kw),
           sos.Scenario(surface="ocean", grd_alb=0.02, wind_speed=5.0, brdf_vol=0.1, **kw)]
    good = sos.Scenario(surface="ocean", grd_alb=0.02, wind_speed=5.0, **kw)
    for sc in bad:
        with pytest.raises(ValueError):
            sos.solve_scenarios([good, sc])
        with pytest.raises(ValueError):
            sos.BatchSolver([sc])
        with pytest.raises(ValueError):
            sos.solve_azimuthal([good, sc], [0.0], 2)


def test_split_at_64_glint_sets():
    scs = [sos.Scenario(nb_layers=60, nb_angles=41, surface="ocean", grd_alb=0.02, wind_speed=0.25 * i) for i in range(70)]
    assert [len(b) for b in DR.split_for_plan_limits(scs, range(70))] == [64, 6]
    same = [dataclasses.replace(sc, wind_speed=5.0) for sc in scs]
    assert [len(b) for b in DR.split_for_plan_limits(same, range(70))] == [70]
    # the azimuthal mode is part of the set: 70 members of one wind speed in 70 modes need two plans
    assert [len(b) for b in DR.split_for_plan_limits(same, range(70), brdf_modes=list(range(70)))] == [64, 6]


def test_solve_azimuthal_accepts_the_ocean(monkeypatch):
    class Reached(Exception):
        pass

    def sentinel(*a, **k):
        raise Reached
    monkeypatch.setattr(AZ, "solved_batches", sentinel)
    sc = sos.Scenario(nb_layers=120, nb_angles=41, surface="ocean", grd_alb=0.02, wind_speed=3.0)
    with pytest.raises(Reached):
        sos.solve_azimuthal([sc], [0.0, np.pi], 3)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    sos._lib.load()
    return torch


def engine_for(M, L=32, region_start=None):
    mu = sos.mu_grid(M)
    tau = np.linspace(0.0, 0.5, L)
    w = sos.grid.extrapolation_width(float(tau[-1]), M)
    sc = sos.ScenarioCoefficients(mu0=0.5, grd_alb=0.02, tauStar_tot=0.5, coef_atm=1.0, extrap_width=(w, w, w))
    return sos.SosEngine(mu, tau[None, :], [sc], region_start=region_start or [0, 8, 16, L], surface=sos._lib.SURFACE_OCEAN)


def ocean_batch(**over):
    base = dict(nb_layers=96, nb_angles=251, atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.5), surface="ocean")
    base.update(over)
    return [sos.Scenario(mu0=0.5, tauStar_atm=0.124, tauStar_aer=0.0, grd_alb=0.02, wind_speed=5.0, **base),
            sos.Scenario(mu0=0.37, tauStar_atm=0.6, tauStar_aer=0.9, alb_aer=0.8, alb_atm=0.9, grd_alb=0.05, wind_speed=1.0,
                         ocean_index=1.33, **base),
            sos.Scenario(mu0=0.9, tauStar_atm=0.3, tauStar_aer=0.2, alb_aer=1.0, grd_alb=0.0, wind_speed=12.0, **base),
            sos.Scenario(mu0=0.2, tauStar_atm=0.05, tauStar_aer=0.01, alb_aer=0.95, grd_alb=0.03, wind_speed=0.0,
                         z_up=60.0, z_down=30.0, **base)]


@pytest.mark.gpu
def test_device_builder_matches_the_reference(gpu):
    for M in (41, 101):
        mu = sos.mu_grid(M)
        eng = engine_for(M)
        try:
            for W in (0.0, 5.0, 15.0):
                for K in (8, 64):
                    R = eng.build_glint_modes(W, 1.34, n_modes=K).cpu().numpy()
                    assert R.shape[:2] == (K, M)
                    want = OC.glint_modes(M, mu, W, 1.34, K)                 # [m][i][c]
                    got = R[:, :, : M - 1].transpose(0, 2, 1)                # [m][c][i] -> [m][i][c]
                    assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want)), (M, W, K)
        finally:
            eng.close()


@pytest.mark.gpu
def test_parity_with_the_oracle_construction(gpu, so):
    wide = sos.Scenario(mu0=0.6, tauStar_atm=0.124, tauStar_aer=0.12, alb_aer=0.97, grd_alb=0.02, wind_speed=7.0,
                        surface="ocean", atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.7))   # the default grid
    for scs in (ocean_batch(), [wide]):
        got = sos.solve_scenarios(scs)
        worst = 0.0
        for i, (sc, r) in enumerate(zip(scs, got)):
            ref, mu = solve_ref(so, sc)
            assert r.n == ref["n"] and r.status == 0, (i, r.n, ref["n"], r.status)
            err = relmax(r.I, ref["I"])
            worst = max(worst, err)
            assert err < TOL and relelem(r.I, ref["I"]) < 1e-8, (i, err)
            assert_quadratures_match(so, sc, r, ref, mu)
        print(f"ocean parity: worst relmax {worst:.2e}")


@pytest.mark.gpu
def test_zero_glint_weight_is_bit_identical_to_the_diffuse_ground(gpu):
    scs = ocean_batch()[:3]   # (one grid group: the fourth has its own aerosol rows)
    bs = sos.BatchSolver(scs)
    try:
        M = bs.M
        sets = np.array([bs._brdf_sets.index(DR._glint_key(sc)) for sc in scs])
        beams = np.zeros((len(scs), 2, M - 1))
        for s, sc in enumerate(scs):
            beams[s, 0] = DR.glint_beam(M, bs.mu, sc, 1)[0]
        bs.engine.set_brdf_scenarios(sets, np.zeros((len(scs), 2)), beams)
        got = bs.results(bs.solve(), quadratures=True)
    finally:
        bs.engine.close()
    want = sos.solve_scenarios([dataclasses.replace(sc, surface="lambert_diffuse", wind_speed=None) for sc in scs])
    for x, y in zip(got, want):
        assert x.n == y.n and x.status == y.status and np.array_equal(x.I, y.I)
        for q in ("flux_up", "flux_down", "net_flux", "diffusivity", "heating_rate"):
            assert np.array_equal(getattr(x, q), getattr(y, q)), q
        assert x.toa_net_flux == y.toa_net_flux


def non_scattering(M=101, W=1.0, mu0=0.3):
    return sos.Scenario(nb_layers=60, nb_angles=M, mu0=mu0, tauStar_atm=0.3, tauStar_aer=0.1, alb_atm=0.0, alb_aer=0.0,
                        grd_alb=0.02, wind_speed=W, max_orders=1, surface="ocean", atm_phase=("rayleigh", 0.0),
                        aer_phase=("hg", 0.5))


def direct_glint(sc, phi):
    """(surface row, TOA row) of E rho(mu, mu0, phi) e^{-(T - tau)/mu} on the upward columns: (n_phi, M-1) each."""
    M = sc.nb_angles
    mu = sos.mu_grid(M)[M + 1:]
    T = sc.tauStar_atm + sc.tauStar_aer
    want = (sc.grd_alb + OC.cox_munk(mu[None, :], sc.mu0, phi[:, None], sc.wind_speed)) * np.exp(-T / sc.mu0)
    return want, want * np.exp(-T / mu)[None, :]


@pytest.mark.gpu
def test_without_scattering_the_radiance_is_the_exact_glint(gpu, monkeypatch):
    """alb = 0, one order, W = 1 m/s: the surface and TOA rows are E rho e^{-(T - tau)/mu} at every phi to 1e-12 of the peak;
    without the correction the 64-mode series is off by several per cent of the peak."""
    sc, K = non_scattering(), 64
    M = sc.nb_angles
    phi = np.linspace(0, np.pi, 181)
    surf, toa = direct_glint(sc, phi)
    a = sos.solve_azimuthal([sc], phi, K, rows=(0, -1), n_quad=2 * K)[0]
    assert np.all(a.mode_orders == 1)
    assert np.max(np.abs(a.radiance[1][:, M + 1:] - surf)) <= 1e-12 * np.max(surf)
    assert np.max(np.abs(a.radiance[0][:, M + 1:] - toa)) <= 1e-12 * np.max(toa)
    assert int(np.argmax(a.radiance[1][:, M + 1 + int(np.argmin(np.abs(sos.mu_grid(M)[M + 1:] - sc.mu0)))])) == 0
    monkeypatch.setattr(sos.SosEngine, "glint_correction", lambda self, out, *args: out)
    b = sos.solve_azimuthal([sc], phi, K, rows=(0, -1), n_quad=2 * K)[0]
    err = np.max(np.abs(b.radiance[1][:, M + 1:] - surf)) / np.max(surf)
    assert err > 0.02, err
    assert np.array_equal(a.modes, b.modes) and np.array_equal(a.base.I, b.base.I)
    print(f"64-mode series without the correction: {err:.3f} of the peak")


@pytest.mark.gpu
def test_azimuth_over_the_ocean(gpu, so):
    """base = solve_scenarios bit for bit; modes 1, 2, 5 are the oracle construction with the glint mode m run for n_0
    orders; an isotropic medium over the sea still has azimuth dependence."""
    from test_azimuth import L_SMALL, M_SMALL
    K = 6
    scs = [sos.Scenario(nb_layers=L_SMALL, nb_angles=M_SMALL, mu0=0.5, tauStar_atm=0.124, tauStar_aer=0.12, grd_alb=0.02,
                        wind_speed=6.0, alb_aer=0.97, atm_phase=("rayleigh", 0.5), aer_phase=("hg", 0.6), surface="ocean"),
           sos.Scenario(nb_layers=L_SMALL, nb_angles=M_SMALL, mu0=0.8, tauStar_atm=0.2, tauStar_aer=0.1, grd_alb=0.0,
                        wind_speed=2.0, ocean_index=1.33, alb_aer=0.9, alb_atm=0.9, atm_phase=("iso", 0.0),
                        aer_phase=("iso", 0.0), surface="ocean")]
    phi = np.arange(2 * K + 3) * (2 * np.pi / (2 * K + 3))
    az = sos.solve_azimuthal(scs, phi, K, rows=tuple(range(L_SMALL)), n_quad=25)
    ref = sos.solve_scenarios(scs)
    mu = sos.mu_grid(M_SMALL)
    for a, r, sc in zip(az, ref, scs):
        assert np.array_equal(a.base.I, r.I) and a.base.n == r.n and a.base.toa_net_flux == r.toa_net_flux
        n0 = r.n
        assert np.all(a.mode_orders == n0) and np.all(a.mode_status == 0), (a.mode_orders, a.mode_status)
        P0a, Pa = sos.phase_modes(sc.atm_phase[0], M_SMALL, mu, K, sc.atm_phase[1], mu0=sc.mu0)
        P0e, Pe = sos.phase_modes(sc.aer_phase[0], M_SMALL, mu, K, sc.aer_phase[1], mu0=sc.mu0)
        osc = oracle_scenario(so, sc, grd_alb=0.0)
        for m in (1, 2, 5):
            gr = glint_ground(M_SMALL, mu, sc.mu0, sc.wind_speed, sc.ocean_index, m, K)
            want = rossli_solve(so, osc, P0a[m], Pa[m], P0e[m], Pe[m], 1.0, 0.0, *gr, n_orders=n0)["I"]
            assert np.max(np.abs(want)) > 0
            assert relmax(a.modes[m], want) <= TOL and relelem(a.modes[m], want) <= 1e-8, m
    assert np.max(np.abs(az[1].modes[1])) > 1e-3 * np.max(np.abs(az[1].modes[0]))   # isotropic medium, azimuth-dependent


@pytest.mark.gpu
def test_plan_reuse_across_wind_speeds_equals_fresh_solvers(gpu):
    first = ocean_batch()[:3]
    second = [dataclasses.replace(sc, mu0=0.3 + 0.2 * i, grd_alb=0.01 * i, wind_speed=2.0 + 4.0 * i, tauStar_atm=0.2 + 0.1 * i)
              for i, sc in enumerate(first)]
    reused = sos.BatchSolver(first)
    try:
        for k, batch in enumerate((first, second)):
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
def test_more_than_64_glint_sets_are_split(gpu, so):
    base = dict(nb_layers=60, nb_angles=41, atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.6), surface="ocean",
                tauStar_atm=0.2, tauStar_aer=0.1, alb_aer=0.9, grd_alb=0.02)
    scs = [sos.Scenario(mu0=0.3 + 0.005 * i, wind_speed=0.2 * i, **base) for i in range(70)]
    got = sos.solve_scenarios(scs)
    for i in (0, 40, 63, 64, 69):
        ref, _ = solve_ref(so, scs[i])
        assert got[i].n == ref["n"] and relmax(got[i].I, ref["I"]) < TOL, i


@pytest.mark.gpu
def test_critical_albedo_sweep_forcing_is_the_toa_difference(gpu):
    base = dict(nb_layers=96, nb_angles=101, atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.7), surface="ocean")
    pts = [sos.Scenario(mu0=0.5, tauStar_atm=0.124, tauStar_aer=0.12, grd_alb=0.02, wind_speed=5.0, **base),
           sos.Scenario(mu0=0.7, tauStar_atm=0.124, tauStar_aer=0.3, grd_alb=0.01, wind_speed=10.0, **base)]
    omega_c, forcing, n_solves, omega = sos.critical_albedo_sweep(pts, return_evaluated=True)
    assert n_solves > len(pts) and np.all(np.isfinite(forcing))
    for p, w, f in zip(pts, omega, forcing):
        with_aer = sos.solve_scenarios([dataclasses.replace(p, alb_aer=float(w))])[0].toa_net_flux
        without = sos.solve_scenarios([dataclasses.replace(p, tauStar_aer=0.0, alb_aer=1.0)])[0].toa_net_flux
        assert abs(f - (with_aer - without)) <= 1e-10 * max(abs(with_aer), abs(without))


@pytest.mark.gpu
def test_plan_refusals(gpu):
    """A single-layer plan refuses the surface (-4); a plan without its glint data answers SOS_ERR_STATE (-5) to a first
    order; the plan takes one matrix per set and a zero second weight (SOS_ERR_INVALID, -1, otherwise)."""
    with pytest.raises(sos._lib.SosError, match=r"\(-4\)"):
        engine_for(41, region_start=[0, 32])
    eng = engine_for(41)
    try:
        with pytest.raises(sos._lib.SosError, match=r"\(-5\)"):
            eng.first_order(np.zeros((1, 2, eng.N)))
        R = eng.build_glint_modes(5.0, n_modes=1)
        with pytest.raises(sos._lib.SosError, match=r"\(-1\)"):
            eng.set_brdf([(R[0], R[0])])
        eng.set_brdf([R[0]])
        beams = np.zeros((1, 2, eng.M - 1))
        with pytest.raises(sos._lib.SosError, match=r"\(-1\)"):
            eng.set_brdf_scenarios(np.zeros(1), np.array([[1.0, 0.5]]), beams)
        beams[0, 1] = np.nan                                                    # the second beam vector is not read
        eng.set_brdf_scenarios(np.zeros(1), np.array([[1.0, 0.0]]), beams)
    finally:
        eng.close()
