"""Azimuth-resolved radiance: Fourier modes of the phase function solved as batch members and summed on the device.

Every field the drivers return is the azimuth average (mode 0) of the radiance.  For a plane-parallel medium each Fourier
mode m of the radiance obeys the same equation as mode 0 -- the same contraction J = (omega/4) int P I dmu', sweeps and
specular mirror coupling -- with the operand P_m and the solar vector P0_m of phase.phase_modes instead of P and P0.  A
diffuse Lambert ground ('lambert_diffuse') is isotropic and enters mode 0 only: modes m >= 1 are solved over a black
ground.  A Ross-Li ground ('rossli') couples mode m through its own kernel modes (brdf module): the members of mode m keep
the surface with grd_alb = 0 (the isotropic part has no mode m >= 1) and the Ross-Li mode m; so do those of an ocean
('ocean') with the glint mode m.  So a
(geometry, mode) pair is one more member of a batch: its own operand index and first-order table row, summing exactly the
orders its mode 0 summed (sos_scenario.order_cap), and

    I(tau, mu, phi) = I_0 + 2 sum_{m >= 1} I_m cos(m phi)

is summed on the device (sos_azimuth_synthesis).  Over an ocean the radiance also gets the once-reflected direct beam in
closed form (sos_glint_correction): the glint lobe is too narrow in azimuth for 64 modes at low wind, so its truncated
series is replaced by the exact reflectance on every upward column.  With single_scatter='exact' the radiance also gets the
singly scattered light in closed form (sos_single_scatter_correction): a K-term series cannot follow a sharply peaked phase
function, and the first order's angular shape is the phase function, so its truncated series is replaced by the closed-form
first order of p(cos Theta) / T at every azimuth (DESIGN section 13).

phi is the azimuth of the PROPAGATION direction of the diffuse light relative to the propagation azimuth of the solar beam:
with the grid's signs (mu < 0 downward) the beam travels along (-mu0, 0), cos Theta = -mu0 mu + sqrt(1 - mu0^2) sqrt(1 - mu^2)
cos phi, and phi = 0 is the forward half-plane.  A sensor's relative azimuth (the azimuth of its viewing direction, opposite
to the propagation of the light it receives) is phi + pi.
"""
from __future__ import annotations

from dataclasses import dataclass, replace
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from . import phase as PH
from . import ocean as OC
from .drivers import (DriverResult, MAX_PHASES_PER_PLAN, BatchSolver, Scenario, _BRDF_STACKS, _GLINT_STACKS, _MODE_STACKS, _PHASES,
                      check_brdf, glint_beam, grid_groups, solved_batches, split_for_plan_limits)

# phase functions per plan of the mode members (two per mode: typically 8 modes per plan)
MODE_PHASES_PER_PLAN = MAX_PHASES_PER_PLAN


@dataclass
class AzimuthalResult:
    """base: the mode-0 result (what solve_scenarios returns for the scenario); radiance (n_rows, n_phi, N): I(tau_row, mu, phi)
    at the layers `rows` and azimuths `phi` (over an ocean with the exact direct glint: the once-reflected, unscattered beam
    in closed form instead of its truncated series); modes (n_modes, n_rows, N): the Fourier components I_m at those layers
    (the truncated series, order for order; mode 0 = base.I rows); mode_orders / mode_status (n_modes,): orders summed and
    status bits of every mode (a mode whose atmosphere and aerosol modes vanish is not solved: 0 orders, I_m = 0);
    single_scatter: 'series' (radiance is the truncated series) or 'exact' (its first order by the phase function is exact)."""
    base: DriverResult
    radiance: np.ndarray
    rows: np.ndarray
    phi: np.ndarray
    n_modes: int
    modes: np.ndarray
    mode_orders: np.ndarray
    mode_status: np.ndarray
    single_scatter: str = "series"


def _mode_spec(spec, m: int, n_quad: int):
    name, g = PH.resolve(spec[0], spec[1] if len(spec) > 1 else None)
    return (name, g, m, n_quad)


def _vanishes(spec, m: int) -> bool:
    return PH.mode_vanishes(PH.resolve(spec[0], spec[1] if len(spec) > 1 else None)[0], m)


SINGLE_SCATTER = ("series", "exact")


def _validate(scenarios: Sequence[Scenario], n_modes: int, n_quad: int, single_scatter: str = "series"):
    check_brdf(scenarios)
    if single_scatter not in SINGLE_SCATTER:
        raise ValueError(f"solve_azimuthal: single_scatter must be one of {SINGLE_SCATTER}, not {single_scatter!r}")
    if n_modes < 1:
        raise ValueError("solve_azimuthal: n_modes must be >= 1")
    if n_quad < 2 * n_modes:
        raise ValueError(f"solve_azimuthal: n_quad = {n_quad} azimuth nodes cannot resolve {n_modes} modes (need >= 2 n_modes)")
    for sc in scenarios:
        if sc.surface in ("lambert", "lambert_readme") and sc.grd_alb > 0:
            # the first order reflects the beam specularly while the n >= 2 coupling is isotropic: no consistent mode split
            raise ValueError(f"solve_azimuthal: surface {sc.surface!r} with grd_alb > 0 has no Fourier-mode decomposition; "
                             "surface='lambert_diffuse' is a Lambertian ground in every order")
        for spec in (sc.atm_phase, sc.aer_phase):
            if not isinstance(spec[0], str):
                raise ValueError("solve_azimuthal: modes are built from the phase function; (P0, P) arrays cannot be split")


def solve_azimuthal(scenarios: Sequence[Scenario], phi, n_modes: int, rows=(0, -1), n_quad: int = 25,
                    device=None, single_scatter: str = "series") -> List[AzimuthalResult]:
    """Radiance as a function of azimuth for every scenario: modes 0 .. n_modes-1, synthesized at the azimuths `phi`
    (radians, see the module docstring for the convention) on the layers `rows` (negative = from the bottom).

    Mode 0 is solved exactly as solve_scenarios solves it (result.base); modes 1 .. n_modes-1 of all geometries are batched
    with order_cap = the orders their mode 0 summed, so the azimuth-resolved field is the same truncated series, order for
    order, as the mode-0 field.  n_quad: azimuth nodes of the mode builder (>= 2 n_modes; 25 = the azimuth-averaged
    builders' nodes, enough for Rayleigh and moderate HG -- sharp peaks need more).  A 'lambert_diffuse' ground enters mode 0
    only (the modes m >= 1 of its geometries are solved over a black ground); a 'rossli' ground enters every mode through
    its kernel modes, which are integrated on brdf.BRDF_NODES nodes whatever n_quad; so does an 'ocean' through its glint
    modes, and its radiance includes the exact direct glint (the once-reflected beam transmitted without scattering, in closed
    form instead of its n_modes-term series; `modes` and `base` stay the truncated series).  'lambert' / 'lambert_readme'
    surfaces with grd_alb > 0 and caller-supplied (P0, P) arrays raise ValueError before any device work.

    single_scatter='exact' replaces the n_modes-term series of the singly scattered radiance (the first order by the phase
    function: the direct beam and, over a specular ground, the mirror-reflected beam) by its closed form with the exact
    p(cos Theta) / T at every azimuth, T the mode-0 normalisation at n_quad nodes (phase.phase_exact).  The surface terms of
    the first order over 'lambert_diffuse', 'rossli' and 'ocean' grounds stay the series; `modes` and `base` do too.  The
    default 'series' returns the truncated series; any other value raises ValueError before any device work."""
    scenarios = list(scenarios)
    K, n_quad = int(n_modes), int(n_quad)
    _validate(scenarios, K, n_quad, single_scatter)
    phi = np.atleast_1d(np.asarray(phi, dtype=np.float64))
    if phi.ndim != 1:
        raise ValueError("solve_azimuthal: phi must be a 1-D sequence of azimuths")
    n_az = phi.size
    for sc in scenarios:
        if not all(-sc.nb_layers <= int(r) < sc.nb_layers for r in rows) or len(rows) == 0:
            raise ValueError(f"solve_azimuthal: rows must lie in [-{sc.nb_layers}, {sc.nb_layers})")
    w_modes = 2.0 * np.cos(np.arange(K)[:, None] * phi[None, :])   # row m >= 1: 2 cos(m phi_p)
    ones = np.ones(n_az)
    out: List[Optional[AzimuthalResult]] = [None] * len(scenarios)
    try:
        for group in grid_groups(scenarios):
            rws = np.array([int(r) for r in rows], dtype=np.int64) % scenarios[group[0]].nb_layers
            pos = {i: k for k, i in enumerate(group)}
            n0 = {}
            base = {}
            modes = {i: np.zeros((K, rws.size, 2 * scenarios[i].nb_angles)) for i in group}
            orders = {i: np.zeros(K, dtype=np.int64) for i in group}
            status = {i: np.zeros(K, dtype=np.int64) for i in group}
            radiance = None
            for idxs, bs, res, results in solved_batches(scenarios, device=device, groups=[group]):
                eng = bs.engine
                if radiance is None:
                    radiance = torch.empty((len(group), rws.size, n_az, eng.N), dtype=torch.float64, device=eng.device)
                eng.azimuth_synthesis(res.I, np.array([pos[i] for i in idxs]), np.tile(ones, (len(idxs), 1)), len(group), rws,
                                      radiance, accumulate=False)
                if scenarios[idxs[0]].surface == "ocean":
                    _glint_correction(eng, bs, [scenarios[i] for i in idxs], [pos[i] for i in idxs], rws, K, phi, radiance)
                if single_scatter == "exact":
                    _single_scatter_correction(eng, bs, [pos[i] for i in idxs], rws, K, n_quad, phi, radiance)
                for i, r in zip(idxs, results):
                    base[i], n0[i] = r, int(r.n)
                    modes[i][0] = r.I[rws]
                    orders[i][0], status[i][0] = r.n, r.status
            # modes 1 .. K-1 of every geometry of the group, each summing the orders of its mode 0
            members, keys = [], []
            for i in group:
                sc = scenarios[i]
                for m in range(1, K):
                    brdf = (sc.surface == "rossli" and (sc.brdf_vol != 0 or sc.brdf_geo != 0)) or sc.surface == "ocean"
                    if _vanishes(sc.atm_phase, m) and _vanishes(sc.aer_phase, m) and not brdf:
                        continue   # I_m = 0: nothing to solve (a Ross-Li or ocean ground reflects mode m of the beam itself)
                    mode_sc = replace(sc, atm_phase=_mode_spec(sc.atm_phase, m, n_quad), aer_phase=_mode_spec(sc.aer_phase, m, n_quad))
                    if sc.surface == "lambert_diffuse":
                        mode_sc = replace(mode_sc, surface="specular", grd_alb=0.0)   # an isotropic ground has no mode m >= 1
                    elif sc.surface in ("rossli", "ocean"):
                        mode_sc = replace(mode_sc, grd_alb=0.0)   # the kernels' / glint's mode m (BatchSolver brdf_modes below)
                    members.append(mode_sc)
                    keys.append((i, m))
            for sub in split_for_plan_limits(members, range(len(members)), max_phases=MODE_PHASES_PER_PLAN,
                                             brdf_modes=[k[1] for k in keys]):
                caps = [n0[keys[j][0]] for j in sub]
                brdf = members[sub[0]].surface in ("rossli", "ocean")
                bs = BatchSolver([members[j] for j in sub], device=device, order_caps=caps,
                                 brdf_modes=[keys[j][1] for j in sub] if brdf else None)
                try:
                    res = bs.solve(max_orders=max(caps))
                    eng = bs.engine
                    geo = np.array([pos[keys[j][0]] for j in sub])
                    w = np.stack([w_modes[keys[j][1]] for j in sub])
                    eng.azimuth_synthesis(res.I, geo, w, len(group), rws, radiance, accumulate=True)
                    fields = res.I.view(eng.S, eng.L, eng.ld)[:, torch.as_tensor(rws, device=eng.device), : eng.N].cpu().numpy()
                    for s, j in enumerate(sub):
                        i, m = keys[j]
                        modes[i][m] = fields[s]
                        orders[i][m], status[i][m] = res.n_orders[s], res.status[s]
                finally:
                    bs.engine.close()
            rad = radiance.cpu().numpy()
            for i in group:
                out[i] = AzimuthalResult(base=base[i], radiance=rad[pos[i]], rows=rws.copy(), phi=phi.copy(), n_modes=K,
                                         modes=modes[i], mode_orders=orders[i], mode_status=status[i],
                                         single_scatter=single_scatter)
    finally:
        _MODE_STACKS.clear()   # the device mode stacks serve the sub-batches of one call
        _BRDF_STACKS.clear()
        _GLINT_STACKS.clear()
    return out  # type: ignore


def _glint_correction(eng, bs: BatchSolver, scs: Sequence[Scenario], geo: Sequence[int], rws: np.ndarray, K: int, phi: np.ndarray,
                      radiance: torch.Tensor):
    """Replace the K-term series of the once-reflected, unscattered direct beam in `radiance` by the exact glint for the
    ocean geometries `scs` of one mode-0 batch (sos_glint_correction); the modes m >= 1 of those geometries are all solved."""
    M = bs.M
    par = np.array([[sc.mu0, sc.tauStar_atm + sc.tauStar_aer, float(OC.slope_variance(sc.wind_speed)), sc.ocean_index]
                    for sc in scs], dtype=np.float64)
    beams = np.stack([glint_beam(M, bs.mu, sc, K) for sc in scs])
    eng.glint_correction(radiance, np.asarray(geo), par, bs.tau[:, rws], beams, phi)


def _single_scatter_correction(eng, bs: BatchSolver, geo: Sequence[int], rws: np.ndarray, K: int, n_quad: int, phi: np.ndarray,
                               radiance: torch.Tensor):
    """Replace the K-term series of the singly scattered radiance in `radiance` by its closed form for the geometries of one
    mode-0 batch (sos_single_scatter_correction).  The subtracted series is made of the vectors the radiance was summed with:
    mode 0 the batch's own P0 table row, modes m >= 1 the mode members' (the host-built _PHASES entries, exact zeros for a
    vanishing mode); an isotropic phase function has no correction."""
    M, mu = bs.M, bs.mu
    ents, vecs, vec_row, tabs, tab_off = [], [], {}, [], {}
    n_tab = 0
    for s, sc in enumerate(bs.scenarios):
        e = np.zeros((), dtype=_lib.SS_ENTRY_DTYPE)
        e["scenario"], e["geo"], e["w"] = s, geo[s], bs.P0w[s]
        for j, spec in enumerate((sc.atm_phase, sc.aer_phase)):
            name, g = PH.resolve(spec[0], spec[1] if len(spec) > 1 else None)
            if name == "iso":
                e["family"][j] = -1
                continue
            e["family"][j] = PH.FAMILY_CODE[name]
            key = (name, tuple(g) if isinstance(g, (tuple, list)) else float(g), float(sc.mu0))
            if key not in vec_row:
                v = np.empty((K, bs.N))
                v[0] = bs.P0tab[bs.P0idx[s, j]]
                for m in range(1, K):
                    v[m] = 0.0 if PH.mode_vanishes(name, m) else _PHASES.get(_mode_spec(spec, m, n_quad), M, mu, sc.mu0, need_P=False)[0]
                vec_row[key] = (len(vecs), PH.exact_norm(name, mu, sc.mu0, g, n_quad))
                vecs.append(v)
            e["series"][j], e["norm"][j] = vec_row[key]
            if name in PH.TABULATED:
                if key[:2] not in tab_off:
                    xs, ys = PH.phase_table(name, g)
                    tab_off[key[:2]] = (n_tab, len(xs))
                    tabs += [np.asarray(xs, dtype=np.float64), np.asarray(ys, dtype=np.float64)]
                    n_tab += 2 * len(xs)
                e["tab_off"][j], e["tab_n"][j] = tab_off[key[:2]]
            else:
                e["g"][j] = float(g)
        if not np.all(e["family"] < 0):
            ents.append(e)
    if not ents:
        return   # isotropic media: the series is exact
    eng.single_scatter_correction(radiance, np.array(ents, dtype=_lib.SS_ENTRY_DTYPE), np.stack(vecs),
                                  np.concatenate(tabs) if tabs else np.zeros(0), rws, phi)
