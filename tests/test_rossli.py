"""surface="rossli": a Ross-Li bidirectional ground (RossThick + LiSparse-R kernels) in every order and azimuthal mode.

rho = f_iso + f_vol K_vol + f_geo K_geo.  The f_iso part is the 'lambert_diffuse' coupling unchanged; every upward column i
of the surface row adds

    order 1:  sum_k f_k (e^{-T/mu0} beta_k[i] + sum_c u_c R^k[i][c])        order n:  sum_k f_k sum_c u_c R^k[i][c]

with u_c = -2 w_c mu_c I_n[L-1, c] (w: trapezoid weights of the ascending downward half), R^k the kernels' mode matrices
(brdf.brdf_modes) and beta_k the beam vectors (brdf.brdf_beam).  The oracle has no such surface; `rossli_solve` below
builds it from the oracle's own pieces, as test_lambert_diffuse.py does for the diffuse Lambert ground: the black-ground
first order plus the per-column surface radiance, then order_sweeps, whose mirror branch forms its seed as
`grd_alb * I_n[L-1, M-2::-1]` -- `RossLiSeed` stands in for grd_alb there and returns the Ross-Li seed of that row.
"""
import dataclasses
from importlib import import_module

import numpy as np
import pytest

from conftest import relelem, relmax
from test_lambert_diffuse import (TOL, IDENTITY_KW, assert_quadratures_match, diffuse_solve, identity_phases, no_blend,
                                  oracle_scenario)

import sos_b200 as sos

BR = sos.brdf
AZ = import_module("sos-radiative-transfer_b200.azimuth")


@pytest.fixture(scope="module")
def so():
    import sos_oracle
    return sos_oracle


def down_weights(mu, M):
    """-2 w_c mu_c over the downward half (u = this * I[L-1, :M])."""
    x = mu[:M]
    hi = np.append(x[1:], x[-1])
    lo = np.insert(x[:-1], 0, x[0])
    return -2.0 * (0.5 * (hi - lo)) * x


class RossLiSeed:
    """grd_alb of the oracle's mirror branch: `self * I_n[L-1, M-2::-1]` is the Ross-Li seed of the upward columns."""

    def __init__(self, so, rho, fv, fg, Rv, Rg, mu, M):
        self.so, self.rho, self.fv, self.fg, self.Rv, self.Rg, self.mu, self.M = so, rho, fv, fg, Rv, Rg, mu, M

    def seed(self, row):
        mu, M = self.mu, self.M
        ell = -2 * self.rho * self.so.trapz(row * mu[:M], mu[:M])
        u = down_weights(mu, M) * row
        return ell + (self.fv * (self.Rv @ u) + self.fg * (self.Rg @ u))

    def __mul__(self, mirrored):
        return self.seed(np.append(mirrored[::-1], 0.0))   # I_n[L-1, 0 .. M-1]; column M-1 (mu = 0-) has the weight mu = 0


def rossli_first_order(so, osc, tau, mu, iu, idn, P0a, P0e, fv, fg, Rv, Rg, bv, bg):
    """Order 1 over the Ross-Li ground and its per-column surface radiance b."""
    M, L = osc.nb_angles, osc.nb_layers
    I1 = so.first_order_regions(dataclasses.replace(osc, grd_alb=0.0, surface="specular"), tau, mu, iu, idn, P0a, P0e)
    T = osc.tauStar_atm + osc.tauStar_aer
    E = np.exp(-T / osc.mu0)
    row = I1[L - 1, :M]
    b_s = osc.grd_alb * (E - 2 * so.trapz(row * mu[:M], mu[:M]))
    u = down_weights(mu, M) * row
    b = b_s + (fv * (E * bv + Rv @ u) + fg * (E * bg + Rg @ u))
    up = np.arange(M + 1, 2 * M)
    I1[:, up] += b[None, :] * np.exp(-(tau[L - 1] - tau)[:, None] / mu[up][None, :])
    return I1, b


def rossli_solve(so, osc, P0a, Pa, P0e, Pe, fv, fg, Rv, Rg, bv, bg, keep_orders=False, n_orders=None):
    """diffuse_solve with the Ross-Li ground; n_orders: sum exactly that many orders (no ratio test)."""
    tau, z, iu, idn = osc.geometry()
    M, L = osc.nb_angles, osc.nb_layers
    mu = so.mu_grid(M)
    I1, b = rossli_first_order(so, osc, tau, mu, iu, idn, P0a, P0e, fv, fg, Rv, Rg, bv, bg)
    lay = so.driver_layout(osc, tau, mu, iu, idn)
    lay.surface, lay.grd_alb = "specular", RossLiSeed(so, osc.grd_alb, fv, fg, Rv, Rg, mu, M)
    dtau_aer = osc.tauStar_aer / (idn + 1 - iu)
    dtau_atm = osc.tauStar_atm / L
    f_atm, f_aer = dtau_atm / (dtau_atm + dtau_aer), dtau_aer / (dtau_atm + dtau_aer)
    A_atm = so.contraction_matrix(Pa, mu, osc.alb_atm)
    A_mix = f_atm * A_atm + f_aer * so.contraction_matrix(Pe, mu, osc.alb_aer)
    In_1, I, In, n, saved = I1, I1.copy(), np.ones_like(I1), 1, [I1]
    while True:
        if n_orders is not None:
            if n >= n_orders:
                break
        else:
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


def ground(M, mu, mu0, m=0, K=None):
    """(Rv, Rg, bv, bg) of mode m, the NumPy reference."""
    K = m + 1 if K is None else K
    Rv, Rg = BR.brdf_modes("vol", M, mu, K)[m], BR.brdf_modes("geo", M, mu, K)[m]
    bv, bg = BR.brdf_beam("vol", M, mu, mu0, K)[m], BR.brdf_beam("geo", M, mu, mu0, K)[m]
    return Rv, Rg, bv, bg


def solve_ref(so, sc, gr=None, **kw):
    M = sc.nb_angles
    mu = so.mu_grid(M)
    P0a, Pa = sos.phase_matrices(sc.atm_phase[0], M, mu, sc.mu0, sc.atm_phase[1])
    P0e, Pe = sos.phase_matrices(sc.aer_phase[0], M, mu, sc.mu0, sc.aer_phase[1])
    gr = ground(M, mu, sc.mu0) if gr is None else gr
    return rossli_solve(so, oracle_scenario(so, sc), P0a, Pa, P0e, Pe, sc.brdf_vol, sc.brdf_geo, *gr, **kw), mu


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_kernel_values():
    kv, kg = BR.rossli_kernels(1.0, 1.0, 0.0)
    assert kv == 0 and kg == 0                                        # nadir / nadir
    mu = np.array([0.95, 0.7, 0.4, 0.15])
    kv, kg = BR.rossli_kernels(mu, mu, 0.0)                           # hot spot: K_geo = sec^2 - sec
    assert np.max(np.abs(kg - (1 / mu ** 2 - 1 / mu))) <= 1e-13 * np.max(1 / mu ** 2)
    rng = np.random.default_rng(3)
    a, b, psi = rng.uniform(0.05, 1, 200), rng.uniform(0.05, 1, 200), rng.uniform(-np.pi, np.pi, 200)
    for x, y in zip(BR.rossli_kernels(a, b, psi), BR.rossli_kernels(b, a, psi)):
        assert np.array_equal(x, y)                                   # reciprocal


def test_mode_matrices_are_reciprocal():
    M, K = 31, 5
    mu = sos.mu_grid(M)
    for kernel in BR.KERNELS:
        R = BR.brdf_modes(kernel, M, mu, K)
        assert R.shape == (K, M - 1, M)
        # R[m][i][c] = rho_m(mu[M+1+i], |mu[c]|) and |mu[c]| = mu[M+1+(M-2-c)]: swap the two cosines
        swapped = R[:, :, : M - 1][:, ::-1, ::-1].transpose(0, 2, 1)
        assert np.max(np.abs(R[:, :, : M - 1] - swapped)) <= 1e-15 * np.max(np.abs(R)), kernel


def test_mode_convention_is_the_ross_li_modes_with_alternating_sign():
    """rho_m = (-1)^m rho_m^{RL}, the Ross-Li modes integrated over psi in [0, pi] directly."""
    K, nq = 8, BR.BRDF_NODES
    a, b = np.array([0.3, 0.55, 0.9]), np.array([0.8, 0.55, 0.2])
    psi = np.linspace(0, np.pi, nq)
    w = np.full(nq, np.pi / (nq - 1))
    w[0] = w[-1] = w[0] / 2
    cm = np.cos(np.arange(K)[:, None] * psi[None, :]) * w[None, :] / np.pi
    for k, kernel in enumerate(BR.KERNELS):
        rl = np.stack([cm @ BR.rossli_kernels(a[j], b[j], psi)[k] for j in range(a.size)], axis=1)
        eng = BR._modes(a, b, K, nq)[k]
        sign = (-1.0) ** np.arange(K)[:, None]
        assert np.max(np.abs(eng - sign * rl)) <= 1e-13 * np.max(np.abs(rl)), kernel


def test_synthesis_reproduces_the_kernels_outside_the_overlap_region():
    """Where the LiSparse overlap vanishes K_geo is a degree-1 trigonometric polynomial in phi; K_vol is smooth."""
    K = 64
    phi = np.linspace(0, np.pi, 17)
    for mi, mv in ((0.3, 0.9), (0.2, 0.7), (1.0, 0.5)):
        modes = BR._modes(np.array([mi]), np.array([mv]), K, BR.BRDF_NODES)[:, :, 0]
        direct = BR.rossli_kernels(mi, mv, phi - np.pi)
        for k in range(2):
            assert np.max(np.abs(BR.brdf_synthesis(modes[k], phi) - direct[k])) <= 1e-12, (mi, mv, k)


def construction(so, rho, fv, fg, **kw):
    M = IDENTITY_KW["nb_angles"]
    mu, ph = identity_phases(M, IDENTITY_KW["mu0"])
    osc = oracle_scenario(so, None, surface="rossli", grd_alb=rho, **IDENTITY_KW)
    return rossli_solve(so, osc, *ph, fv, fg, *ground(M, mu, IDENTITY_KW["mu0"]), **kw), mu, ph


def test_isotropic_weight_alone_is_the_diffuse_lambert_ground(so):
    got, _, ph = construction(so, 0.3, 0.0, 0.0)
    want = diffuse_solve(so, oracle_scenario(so, None, surface="lambert_diffuse", grd_alb=0.3, **IDENTITY_KW), *ph)
    assert got["n"] == want["n"] and np.array_equal(got["I"], want["I"])


def test_zero_weights_are_the_black_ground(so):
    got, _, ph = construction(so, 0.0, 0.0, 0.0)
    want = so.solve(oracle_scenario(so, None, surface="specular", grd_alb=0.0, **IDENTITY_KW), *ph, method="recurrence",
                    use_gemm=True, keep_orders=False)
    assert got["n"] == want["n"] and np.array_equal(got["I"], want["I"])


def test_per_order_seeds_and_order_one(so, monkeypatch):
    """Order 1's surface row is b; order n's upward surface row is f_vol R^vol u_n + f_geo R^geo u_n + l_n of its own
    downward half."""
    no_blend(monkeypatch, so)
    rho, fv, fg = 0.2, 0.15, 0.05
    ref, mu, _ = construction(so, rho, fv, fg, keep_orders=True)
    M, L = IDENTITY_KW["nb_angles"], IDENTITY_KW["nb_layers"]
    Rv, Rg, _, _ = ground(M, mu, IDENTITY_KW["mu0"])
    assert ref["n"] > 3
    assert np.array_equal(ref["I_saved"][0][L - 1, M + 1:], ref["b"])
    assert np.ptp(ref["b"]) > 0.05 * np.max(ref["b"])                 # not isotropic
    for In in ref["I_saved"][1:]:
        row = In[L - 1, :M]
        u = down_weights(mu, M) * row
        ell = -2 * rho * so.trapz(row * mu[:M], mu[:M])
        want = fv * (Rv @ u) + fg * (Rg @ u) + ell
        assert np.max(np.abs(In[L - 1, M + 1:] - want)) <= 1e-14 * np.max(np.abs(want))


def test_refusals_before_any_device_work():
    kw = dict(nb_layers=60, nb_angles=41)
    bad = [sos.Scenario(surface="rossli", grd_alb=0.1, brdf_vol=-0.1, **kw),
           sos.Scenario(surface="rossli", grd_alb=0.1, brdf_geo=float("nan"), **kw),
           sos.Scenario(surface="lambert_diffuse", grd_alb=0.1, brdf_vol=0.1, **kw),
           sos.Scenario(surface="specular", grd_alb=0.1, brdf_geo=0.2, **kw)]
    good = sos.Scenario(surface="rossli", grd_alb=0.1, brdf_vol=0.1, brdf_geo=0.05, **kw)
    for sc in bad:
        with pytest.raises(ValueError):
            sos.solve_scenarios([good, sc])
        with pytest.raises(ValueError):
            sos.BatchSolver([sc])
        with pytest.raises(ValueError):
            sos.solve_azimuthal([good, sc], [0.0], 2)


def test_solve_azimuthal_accepts_the_rossli_ground(monkeypatch):
    class Reached(Exception):
        pass

    def sentinel(*a, **k):
        raise Reached
    monkeypatch.setattr(AZ, "solved_batches", sentinel)
    sc = sos.Scenario(nb_layers=120, nb_angles=41, surface="rossli", grd_alb=0.1, brdf_vol=0.05, brdf_geo=0.02)
    with pytest.raises(Reached):
        sos.solve_azimuthal([sc], [0.0, np.pi], 3)


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    sos._lib.load()
    return torch


def engine_for(M, L=32):
    mu = sos.mu_grid(M)
    tau = np.linspace(0.0, 0.5, L)
    w = sos.grid.extrapolation_width(float(tau[-1]), M)
    sc = sos.ScenarioCoefficients(mu0=0.5, grd_alb=0.1, tauStar_tot=0.5, coef_atm=1.0, extrap_width=(w, w, w))
    return sos.SosEngine(mu, tau[None, :], [sc], region_start=[0, 8, 16, L], surface=sos._lib.SURFACE_ROSSLI)


def rossli_batch(**over):
    base = dict(nb_layers=96, nb_angles=251, atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.5), surface="rossli")
    base.update(over)
    return [sos.Scenario(mu0=0.5, tauStar_atm=0.124, tauStar_aer=0.0, grd_alb=0.15, brdf_vol=0.08, brdf_geo=0.03, **base),
            sos.Scenario(mu0=0.37, tauStar_atm=0.6, tauStar_aer=0.9, alb_aer=0.8, alb_atm=0.9, grd_alb=0.3, brdf_vol=0.2,
                         brdf_geo=0.06, **base),
            sos.Scenario(mu0=0.9, tauStar_atm=0.3, tauStar_aer=0.2, alb_aer=1.0, grd_alb=0.05, brdf_vol=0.0, brdf_geo=0.1, **base),
            sos.Scenario(mu0=0.2, tauStar_atm=0.05, tauStar_aer=0.01, alb_aer=0.95, grd_alb=0.25, brdf_vol=0.12, brdf_geo=0.0,
                         z_up=60.0, z_down=30.0, **base)]


@pytest.mark.gpu
def test_device_builder_matches_the_reference(gpu):
    for M, K in ((41, 6), (251, 3)):
        eng = engine_for(M)
        try:
            R = eng.build_brdf_modes(n_modes=K).cpu().numpy()
        finally:
            eng.close()
        assert R.shape[:3] == (2, K, M)
        mu = sos.mu_grid(M)
        for k, kernel in enumerate(BR.KERNELS):
            want = BR.brdf_modes(kernel, M, mu, K)                      # [m][i][c]
            got = R[k][:, :, : M - 1].transpose(0, 2, 1)                  # [m][c][i] -> [m][i][c]
            assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want)), (M, kernel)


@pytest.mark.gpu
def test_parity_with_the_oracle_construction(gpu, so):
    wide = sos.Scenario(mu0=0.6, tauStar_atm=0.124, tauStar_aer=0.12, alb_aer=0.97, grd_alb=0.12, brdf_vol=0.07, brdf_geo=0.02,
                        surface="rossli", atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.7))   # the default grid
    scs = rossli_batch() + [wide]
    got = sos.solve_scenarios(scs)
    worst = 0.0
    for i, (sc, r) in enumerate(zip(scs, got)):
        ref, mu = solve_ref(so, sc)
        assert r.n == ref["n"] and r.status == 0, (i, r.n, ref["n"], r.status)
        err = relmax(r.I, ref["I"])
        worst = max(worst, err)
        assert err < TOL and relelem(r.I, ref["I"]) < 1e-8, (i, err)
        assert_quadratures_match(so, sc, r, ref, mu)
    print(f"rossli parity: worst relmax {worst:.2e}")


@pytest.mark.gpu
def test_isotropic_weight_alone_is_bit_identical_to_the_diffuse_ground(gpu):
    scs = [dataclasses.replace(sc, brdf_vol=0.0, brdf_geo=0.0) for sc in rossli_batch()]
    pairs = [(scs, [dataclasses.replace(sc, surface="lambert_diffuse") for sc in scs]),
             ([dataclasses.replace(sc, grd_alb=0.0) for sc in scs],
              [dataclasses.replace(sc, grd_alb=0.0, surface="specular") for sc in scs])]
    for a_in, b_in in pairs:
        for x, y in zip(sos.solve_scenarios(a_in), sos.solve_scenarios(b_in)):
            assert x.n == y.n and x.status == y.status and np.array_equal(x.I, y.I)
            for q in ("flux_up", "flux_down", "net_flux", "diffusivity", "heating_rate"):
                assert np.array_equal(getattr(x, q), getattr(y, q)), q
            assert x.toa_net_flux == y.toa_net_flux


@pytest.mark.gpu
def test_without_scattering_the_surface_row_is_the_brdf(gpu):
    """alb = 0, one order: I(tau*, mu, phi) = rho(mu, mu0, phi) e^{-T/mu0} and I(0, mu, phi) = that times e^{-T/mu}."""
    M, K, mu0 = 101, 64, 0.3
    sc = sos.Scenario(nb_layers=60, nb_angles=M, mu0=mu0, tauStar_atm=0.3, tauStar_aer=0.1, alb_atm=0.0, alb_aer=0.0,
                      grd_alb=0.1, brdf_vol=0.3, brdf_geo=0.08, max_orders=1, surface="rossli",
                      atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.5))
    phi = np.linspace(0, np.pi, 13)
    a = sos.solve_azimuthal([sc], phi, K, rows=(0, -1), n_quad=2 * K)[0]
    mu = sos.mu_grid(M)
    T = sc.tauStar_atm + sc.tauStar_aer
    E = np.exp(-T / mu0)
    # columns without LiSparse overlap for any phi (the overlap is smallest at the hot spot: 2 |tan - tan0| >= sec + sec0)
    tan = lambda x: np.sqrt(1 - x * x) / x
    cols = [c for c in range(M + 1, 2 * M)
            if mu[c] > BR.BRDF_MU_MIN and 2 * abs(tan(mu[c]) - tan(mu0)) >= 1 / mu[c] + 1 / mu0]
    assert len(cols) >= 10
    kv, kg = BR.rossli_kernels(mu[cols][None, :], mu0, phi[:, None] - np.pi)
    want = (sc.grd_alb + sc.brdf_vol * kv + sc.brdf_geo * kg) * E                                      # (n_phi, cols)
    surf, toa = a.radiance[1][:, cols], a.radiance[0][:, cols]
    assert np.max(np.abs(surf - want)) <= 1e-11 * np.max(want)
    assert np.max(np.abs(toa - want * np.exp(-T / mu[cols])[None, :])) <= 1e-11 * np.max(want)
    c0 = M + 1 + int(np.argmin(np.abs(mu[M + 1:] - mu0)))
    assert int(np.argmax(a.radiance[1][:, c0])) == phi.size - 1        # the hot spot is at phi = pi


@pytest.mark.gpu
def test_azimuth_over_the_rossli_ground(gpu, so):
    """base = solve_scenarios bit for bit; modes 1, 2, 5 are the oracle construction with the BRDF mode m run for n_0
    orders; an isotropic medium over the ground still has azimuth dependence."""
    from test_azimuth import L_SMALL, M_SMALL
    K = 6
    scs = [sos.Scenario(nb_layers=L_SMALL, nb_angles=M_SMALL, mu0=0.5, tauStar_atm=0.124, tauStar_aer=0.12, grd_alb=0.1,
                        brdf_vol=0.2, brdf_geo=0.05, alb_aer=0.97, atm_phase=("rayleigh", 0.5), aer_phase=("hg", 0.6),
                        surface="rossli"),
           sos.Scenario(nb_layers=L_SMALL, nb_angles=M_SMALL, mu0=0.8, tauStar_atm=0.2, tauStar_aer=0.1, grd_alb=0.2,
                        brdf_vol=0.1, brdf_geo=0.1, alb_aer=0.9, alb_atm=0.9, atm_phase=("iso", 0.0), aer_phase=("iso", 0.0),
                        surface="rossli")]
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
            want = rossli_solve(so, osc, P0a[m], Pa[m], P0e[m], Pe[m], sc.brdf_vol, sc.brdf_geo,
                                *ground(M_SMALL, mu, sc.mu0, m, K), n_orders=n0)["I"]
            assert np.max(np.abs(want)) > 0
            assert relmax(a.modes[m], want) <= TOL and relelem(a.modes[m], want) <= 1e-8, m
        assert relmax(a.radiance.mean(axis=1), a.base.I[a.rows]) <= 1e-13
    assert np.max(np.abs(az[1].modes[1])) > 1e-3 * np.max(np.abs(az[1].modes[0]))   # isotropic medium, azimuth-dependent


@pytest.mark.gpu
def test_plan_reuse_equals_fresh_solvers(gpu):
    first = rossli_batch()[:3]
    second = [dataclasses.replace(sc, mu0=0.3 + 0.2 * i, grd_alb=0.2 - 0.05 * i, brdf_vol=0.05 * i, brdf_geo=0.1 - 0.02 * i,
                                  tauStar_atm=0.2 + 0.1 * i) for i, sc in enumerate(first)]
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
def test_critical_albedo_sweep_forcing_is_the_toa_difference(gpu):
    base = dict(nb_layers=96, nb_angles=101, atm_phase=("rayleigh", 0.0), aer_phase=("hg", 0.7), surface="rossli")
    pts = [sos.Scenario(mu0=0.5, tauStar_atm=0.124, tauStar_aer=0.12, grd_alb=0.15, brdf_vol=0.1, brdf_geo=0.03, **base),
           sos.Scenario(mu0=0.7, tauStar_atm=0.124, tauStar_aer=0.3, grd_alb=0.3, brdf_vol=0.2, brdf_geo=0.05, **base)]
    omega_c, forcing, n_solves, omega = sos.critical_albedo_sweep(pts, return_evaluated=True)
    assert n_solves > len(pts) and np.all(np.isfinite(forcing))
    for p, w, f in zip(pts, omega, forcing):
        with_aer = sos.solve_scenarios([dataclasses.replace(p, alb_aer=float(w))])[0].toa_net_flux
        without = sos.solve_scenarios([dataclasses.replace(p, tauStar_aer=0.0, alb_aer=1.0)])[0].toa_net_flux
        assert abs(f - (with_aer - without)) <= 1e-10 * max(abs(with_aer), abs(without))


@pytest.mark.gpu
def test_single_layer_plan_refuses_the_rossli_ground(gpu):
    E = import_module("sos-radiative-transfer_b200.engine")
    M, L = 41, 32
    mu = sos.mu_grid(M)
    tau = np.linspace(0.0, 0.5, L)
    w = sos.grid.extrapolation_width(float(tau[-1]), M)
    sc = E.ScenarioCoefficients(mu0=0.5, grd_alb=0.3, tauStar_tot=0.5, coef_atm=1.0, extrap_width=(w, w, w))
    with pytest.raises(sos._lib.SosError, match=r"\(-4\)"):
        E.SosEngine(mu, tau[None, :], [sc], region_start=[0, L], surface=sos._lib.SURFACE_ROSSLI)


@pytest.mark.gpu
def test_solve_needs_the_ground_registered(gpu):
    """A Ross-Li plan without its mode matrices and per-scenario data answers SOS_ERR_STATE (-5) to a first order."""
    eng = engine_for(41)
    try:
        C = np.zeros((1, 2, eng.N))
        with pytest.raises(sos._lib.SosError, match=r"\(-5\)"):
            eng.first_order(C)
    finally:
        eng.close()
