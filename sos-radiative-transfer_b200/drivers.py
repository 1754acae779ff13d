"""Three-region drivers: SOS_Aer_main_specular / SOS_Aer_main_lambertian / SOS_Aer_radiative_forcing.

The reference drivers are zero-argument scripts whose parameters are literals inside SOS_Aer()
and whose results are local variables (SOS_Aer_main_specular.py:19-94,478).  Here the same
literals are keyword defaults of `Scenario`, the solve runs on the GPU through libsos_b200 and
the arrays the reference only plots are returned.  Many scenarios that share the grid (layers,
angles, aerosol rows, surface kind) are solved as ONE batch: their fields are stacked along
rows, so the source contraction of every order is a single tall FP64 GEMM.
"""
from __future__ import annotations

from dataclasses import dataclass, field, replace
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib
from . import brdf as BR
from . import ocean as OC
from . import grid as G
from . import phase as PH
from .engine import ScenarioCoefficients, SosEngine

# (name, g), optionally (name, g, m, n_quad): azimuthal Fourier mode m of the family built with n_quad azimuth nodes
# (phase.phase_modes; the azimuth module builds these), or caller-supplied (P0, P) arrays
PhaseSpec = Union[Tuple[str, float], Tuple[str, float, int, int], Tuple[np.ndarray, np.ndarray]]


@dataclass
class Scenario:
    """Parameters of SOS_Aer() with the shipped literals as defaults (SOS_Aer_main_specular.py:23-94)."""
    mu0: float = 0.5
    z0: float = 120.0
    z_up: float = 25.0
    z_down: float = 17.0
    nb_layers: int = 800
    tauStar_atm: float = 0.104
    tauStar_aer: float = 0.120
    grd_alb: float = 1.0
    alb_atm: float = 1.0
    alb_aer: float = 1.0
    nb_angles: int = 501
    atm_phase: PhaseSpec = ("rayleigh", 0.5)
    # the shipped default is the log-normal Mie 'eva' aerosol, which needs miepython; pass explicit
    # (P0, P) arrays for Mie, or an analytic stand-in such as ("hg", 0.5)
    aer_phase: PhaseSpec = ("hg", 0.5)
    # 'specular' | 'lambert' (Lambert-as-coded, SURVEY.md 8c "repair A") | 'lambert_readme' (the n >= 2 coupling with the
    # README's sign and integration range, README.md:215; first order as in the other two: a named physics mode, not parity)
    # | 'lambert_diffuse' (a Lambertian ground in every order: order 1 reflects the direct beam and its own downward light
    # isotropically, no mirror beam; n >= 2 as 'lambert_readme'; the fluxes carry no collimated reflected beam)
    # | 'rossli' (a Ross-Li bidirectional ground in every order, brdf module: grd_alb is f_iso and the 'lambert_diffuse'
    # coupling, brdf_vol / brdf_geo weight the RossThick / LiSparse-R kernels; no collimated reflected beam)
    # | 'ocean' (a wind-roughened sea in every order, ocean module: grd_alb is the isotropic part and the 'lambert_diffuse'
    # coupling, plus the Cox-Munk glint of wind_speed / ocean_index; no collimated reflected beam)
    surface: str = "specular"
    threshold: float = 1e-4
    max_orders: int = 10000
    brdf_vol: float = 0.0   # Ross-Li kernel weights f_vol, f_geo (>= 0; surface='rossli' only)
    brdf_geo: float = 0.0
    wind_speed: Optional[float] = None   # m/s, >= 0 (surface='ocean' only, where it is required)
    ocean_index: float = 1.34            # relative refractive index of the sea (> 1; surface='ocean')


# README scenarios (README.md:95-111) -- tau_atm 0.124, omega_aer 0.97, R_s 0.15
EVA = dict(tauStar_atm=0.124, tauStar_aer=0.120, alb_aer=0.97, grd_alb=0.15, z_up=25.0, z_down=17.0)
WILDFIRE = dict(tauStar_atm=0.124, tauStar_aer=0.0075, alb_aer=0.97, grd_alb=0.15, z_up=15.0, z_down=14.0)


@dataclass
class DriverResult:
    I: np.ndarray
    n: int
    tau: np.ndarray
    mu: np.ndarray
    z_profile: np.ndarray
    idx_up: int
    idx_down: int
    ratio: float
    status: int
    flux_up: Optional[np.ndarray] = None
    flux_down: Optional[np.ndarray] = None
    net_flux: Optional[np.ndarray] = None
    diffusivity: Optional[np.ndarray] = None
    heating_rate: Optional[np.ndarray] = None
    I_saved: Optional[List[np.ndarray]] = None
    toa_net_flux: Optional[float] = None


class PhaseCache:
    """P0/P per (family, g, M, mu0) on the host; P is independent of mu0 and shared."""

    def __init__(self):
        self._P: Dict[tuple, np.ndarray] = {}
        self._P0: Dict[tuple, np.ndarray] = {}

    def get(self, spec: PhaseSpec, M: int, mu: np.ndarray, mu0: float, need_P: bool = True):
        """(P0, P or None, key).  need_P=False skips the host build of the N x N matrix (the caller builds
        it on the device or already holds the operand)."""
        if isinstance(spec[0], str):
            name, g = PH.resolve(spec[0], spec[1] if len(spec) > 1 else None)   # 'eva' / 'wildfire' -> the log-normal Mie mixture
            g = tuple(float(v) for v in g) if isinstance(g, (tuple, list)) else float(g)
            mode = tuple(int(v) for v in spec[2:4]) if len(spec) > 2 else ()   # (m, n_quad) of an azimuthal mode
            kP, k0 = (name, g, M) + mode, (name, g, M, float(mu0)) + mode
            if need_P and kP not in self._P:
                self._P[kP] = PH.phase_P(name, M, mu, g) if not mode else _host_mode(name, g, M, mu, mode)[1]
            if k0 not in self._P0:
                self._P0[k0] = PH.phase_P0(name, M, mu, mu0, g) if not mode else _host_mode(name, g, M, mu, mode, mu0)[0]
            return self._P0[k0], self._P.get(kP), kP
        P0, P = spec
        return np.asarray(P0, dtype=np.float64), np.asarray(P, dtype=np.float64), ("array", id(P))


def _host_mode(name, g, M, mu, mode, mu0=None):
    """(P0_m or None, P_m or None) of mode (m, n_quad) on the host; exact zeros for a mode that vanishes."""
    m, nq = mode
    N = 2 * M
    if PH.mode_vanishes(name, m):
        return (np.zeros(N) if mu0 is not None else None), np.zeros((N, N))
    P0, P = PH.phase_modes(name, M, mu, m + 1, g, mu0=mu0, n_quad=nq, want_P=mu0 is None)
    return (P0[m] if P0 is not None else None), (P[m] if P is not None else None)


_PHASES = PhaseCache()
_MODE_STACKS = {}   # device-built mode stacks (P_0 .. P_{K-1}) per (family, g, grid, n_quad, device), see _DeviceBuilt
_BRDF_STACKS = {}   # device-built Ross-Li mode matrices (2, K, M, ldr) per (grid, device), see BatchSolver._send_brdf
_BRDF_BEAMS = {}    # host beam vectors (2, K, M-1) per (grid, mu0, K)
_GLINT_STACKS = {}  # device-built glint mode matrices (K, M, ldr) per (grid, device, W, n), see BatchSolver._send_brdf
_GLINT_BEAMS = {}   # host glint beam vectors (K, M-1) per (grid, mu0, W, n, K)
_GLINT_STACKS_MAX = 8   # at M = 501 a 64-mode stack is about 130 MB
# surfaces that reflect the direct beam into the diffuse field: the fluxes carry no collimated reflected beam
DIFFUSE_GROUNDS = ("lambert_diffuse", "rossli", "ocean")
MAX_BRDF_SETS_PER_PLAN = 64   # mode matrix sets one plan registers (sosbrdf::MAX_SETS, sos_plan_set_brdf)


def check_brdf(scenarios: Sequence[Scenario]):
    """ValueError for Ross-Li weights that are negative (or not finite) or given on a surface other than 'rossli', and for
    an ocean without a finite wind_speed >= 0 and a finite ocean_index > 1, or a wind_speed on another surface."""
    for sc in scenarios:
        fv, fg = float(sc.brdf_vol), float(sc.brdf_geo)
        if not (np.isfinite(fv) and np.isfinite(fg) and fv >= 0 and fg >= 0):
            raise ValueError(f"Ross-Li kernel weights must be finite and >= 0 (brdf_vol={fv}, brdf_geo={fg})")
        if sc.surface != "rossli" and (fv != 0 or fg != 0):
            raise ValueError(f"brdf_vol / brdf_geo weight the Ross-Li kernels: surface={sc.surface!r} takes none "
                             "(use surface='rossli')")
        if sc.surface == "ocean":
            W, n = sc.wind_speed, float(sc.ocean_index)
            if W is None or not (np.isfinite(float(W)) and float(W) >= 0):
                raise ValueError(f"surface='ocean' needs a finite wind_speed >= 0 in m/s (wind_speed={W})")
            if not (np.isfinite(n) and n > 1):
                raise ValueError(f"surface='ocean' needs a finite ocean_index > 1 (ocean_index={n})")
        elif sc.wind_speed is not None:
            raise ValueError(f"wind_speed drives the ocean glint: surface={sc.surface!r} takes none (use surface='ocean')")


def _glint_key(sc: Scenario, m: int = 0):
    """The glint mode matrix set of an ocean scenario coupled in azimuthal mode m: (W, n, m)."""
    return (float(sc.wind_speed), float(sc.ocean_index), int(m))


def glint_beam(M: int, mu: np.ndarray, sc: Scenario, n_modes: int) -> np.ndarray:
    """The scenario's glint beam vectors of modes 0 .. n_modes-1, (n_modes, M-1) (ocean.glint_beam, cached)."""
    key = (M, float(sc.mu0), float(sc.wind_speed), float(sc.ocean_index), int(n_modes))
    b = _GLINT_BEAMS.get(key)
    if b is None:
        if len(_GLINT_BEAMS) >= 4096:
            _GLINT_BEAMS.clear()
        b = _GLINT_BEAMS[key] = OC.glint_beam(M, mu, sc.mu0, sc.wind_speed, sc.ocean_index, n_modes)
    return b


def clear_caches(disk: bool = False):
    """Forget everything the process keeps between solves: host phase tables, device-resident contraction operands and
    their folded / low-rank companions, the drop-in API's engines (what a cold start pays for again; bench.py's
    e2e_cold).  disk=True also removes the parameter-keyed Mie tables from mie.cache_dir()."""
    from . import api, engine as E, mie
    global _PHASES
    _PHASES._P.clear()
    _PHASES._P0.clear()
    api.clear_cache()
    for d in (E._OPERANDS, E._FOLDED, E._LOWRANK, _BRDF_STACKS, _BRDF_BEAMS, _GLINT_STACKS, _GLINT_BEAMS):
        d.clear()
    mie.lognormal_table.cache_clear()
    if disk:
        import glob
        import os
        for f in glob.glob(os.path.join(mie.cache_dir(), "mie_lognormal_*.npy")):
            try:
                os.remove(f)
            except OSError:
                pass


class _DeviceBuilt:
    """Placeholder for a phase matrix that SosEngine.set_phase builds on the device when (and only
    when) the operand cache misses."""

    def __init__(self, engine, name, g, mode=None):
        self.engine, self.name, self.g, self.mode = engine, name, g, mode

    def build(self):
        if self.mode is None:
            return self.engine.build_phase_matrix(self.name, self.g)[0]
        m, nq = self.mode
        eng = self.engine
        if PH.mode_vanishes(self.name, m):
            return torch.zeros((eng.N, eng.N), dtype=torch.float64, device=eng.device)
        # one launch builds modes 0 .. K-1 together (the phase function is evaluated once per element and node): build in
        # steps of 8 modes and keep the stack for the other modes of the same family
        key = (self.name, self.g, eng.N, eng.mu.tobytes(), nq, eng.device.index)
        stack = _MODE_STACKS.get(key)
        if stack is None or stack.shape[0] <= m:
            stack = _MODE_STACKS[key] = eng.build_phase_modes(self.name, self.g, n_modes=min(64, (m // 8 + 1) * 8), n_quad=nq)[0]
        return stack[m]


def _group_key(sc: Scenario):
    _, iu, idn = G.aerosol_rows(sc.z0, sc.z_up, sc.z_down, sc.nb_layers)
    return (sc.nb_layers, sc.nb_angles, iu, idn, sc.surface)


class BatchSolver:
    """All scenarios of one group (same L, M, aerosol rows, surface) on one device."""

    def __init__(self, scenarios: Sequence[Scenario], device=None, chunk_rows: int = 0, phases: Optional[PhaseCache] = None,
                 device_phase: bool = True, fold: Optional[bool] = None, order_caps: Optional[Sequence[int]] = None,
                 brdf_modes: Optional[Sequence[int]] = None):
        """order_caps: per scenario, sum exactly orders 1 .. cap instead of stopping on the threshold (0 = the threshold;
        sos_scenario.order_cap); None = all 0.  brdf_modes (surface 'rossli' or 'ocean'): per scenario, the azimuthal Fourier
        mode of the Ross-Li kernels or of the glint it is coupled with (0 .. 63; None = all 0, the azimuth average).  An ocean
        batch registers one glint matrix set per distinct (wind_speed, ocean_index, mode): at most 64
        (split_for_plan_limits cuts larger groups).  update() takes both for the next batch the same way."""
        keys = {_group_key(s) for s in scenarios}
        if len(keys) != 1:
            raise ValueError("BatchSolver: scenarios must share nb_layers, nb_angles, aerosol rows and surface")
        self._key = next(iter(keys))
        L, M, self.idx_up, self.idx_down, surf = self._key
        self.L, self.M, self.N = L, M, 2 * M
        self.mu = G.mu_grid(M)
        self._phases = phases or _PHASES
        self._device_phase = device_phase
        self.z = G.aerosol_rows(scenarios[0].z0, scenarios[0].z_up, scenarios[0].z_down, L)[0]
        self._mat_index, self._mats, self._mat_keys = {}, [], []
        coefs = self._prepare(scenarios, order_caps)
        surface = {"specular": _lib.SURFACE_SPECULAR, "lambert": _lib.SURFACE_LAMBERT,
                   "lambert_readme": _lib.SURFACE_LAMBERT_README, "lambert_diffuse": _lib.SURFACE_LAMBERT_DIFFUSE,
                   "rossli": _lib.SURFACE_ROSSLI, "ocean": _lib.SURFACE_OCEAN}[surf]
        self.engine = SosEngine(self.mu, self.tau, coefs, [0, self.idx_up, self.idx_down + 1, L], surface,
                                device=device, chunk_rows=chunk_rows, fold=fold)
        self._register_phases()
        self._brdf_sets = None
        if surf in ("rossli", "ocean"):
            self._send_brdf(brdf_modes)
        self.I1 = None

    def _send_brdf(self, brdf_modes):
        """Ross-Li / ocean plan: register the mode matrix sets the batch uses (when they change) and send every scenario's
        set index, weights and beam vectors."""
        S, M = len(self.scenarios), self.M
        modes = np.zeros(S, dtype=np.int64) if brdf_modes is None else np.asarray(brdf_modes, dtype=np.int64)
        if modes.shape != (S,) or np.any(modes < 0) or np.any(modes >= 64):
            raise ValueError("BatchSolver: brdf_modes must give one mode in [0, 64) per scenario")
        if self._key[4] == "ocean":
            return self._send_glint(modes)
        wanted = sorted(set(modes.tolist()))
        K = wanted[-1] + 1
        eng = self.engine
        if self._brdf_sets is None or not set(wanted) <= set(self._brdf_sets):
            key = (eng.mu.tobytes(), eng.device.index)
            stack = _BRDF_STACKS.get(key)
            if stack is None or stack.shape[1] < K:
                if len(_BRDF_STACKS) >= 4:
                    _BRDF_STACKS.pop(next(iter(_BRDF_STACKS)))
                stack = _BRDF_STACKS[key] = eng.build_brdf_modes(n_modes=K if K == 1 else min(64, (K + 7) // 8 * 8))
            eng.set_brdf([(stack[0, m], stack[1, m]) for m in wanted])
            self._brdf_sets = wanted
        index = {m: j for j, m in enumerate(self._brdf_sets)}
        beams = np.empty((S, 2, M - 1))
        for s, sc in enumerate(self.scenarios):
            bkey = (M, float(sc.mu0), K)
            b = _BRDF_BEAMS.get(bkey)
            if b is None:
                if len(_BRDF_BEAMS) >= 4096:
                    _BRDF_BEAMS.clear()
                b = _BRDF_BEAMS[bkey] = np.stack([BR.brdf_beam(k, M, self.mu, sc.mu0, K) for k in BR.KERNELS])
            beams[s] = b[:, modes[s]]
        eng.set_brdf_scenarios(np.array([index[m] for m in modes.tolist()]),
                               np.array([[sc.brdf_vol, sc.brdf_geo] for sc in self.scenarios], dtype=np.float64), beams)

    def _send_glint(self, modes):
        """Ocean plan: one glint matrix per distinct (W, n, mode) of the batch, weights (1, 0) and the glint beam vectors."""
        S, M = len(self.scenarios), self.M
        keys = [_glint_key(sc, m) for sc, m in zip(self.scenarios, modes.tolist())]
        wanted = sorted(set(keys))
        if len(wanted) > MAX_BRDF_SETS_PER_PLAN:
            raise ValueError(f"BatchSolver: {len(wanted)} distinct (wind_speed, ocean_index, mode) glint sets; one plan "
                             f"takes {MAX_BRDF_SETS_PER_PLAN} (split_for_plan_limits cuts the batch)")
        eng = self.engine
        if self._brdf_sets is None or not set(wanted) <= set(self._brdf_sets):
            need = {}
            for W, n, m in wanted:
                need[(W, n)] = max(need.get((W, n), 0), m + 1)
            stacks = {}
            for (W, n), K in need.items():
                key = (eng.mu.tobytes(), eng.device.index, W, n)
                stack = _GLINT_STACKS.get(key)
                if stack is None or stack.shape[0] < K:
                    if len(_GLINT_STACKS) >= _GLINT_STACKS_MAX:
                        _GLINT_STACKS.pop(next(iter(_GLINT_STACKS)))   # (a registered set keeps its stack alive in the engine)
                    stack = _GLINT_STACKS[key] = eng.build_glint_modes(W, n, n_modes=K if K == 1 else min(64, (K + 7) // 8 * 8))
                stacks[(W, n)] = stack
            eng.set_brdf([stacks[(W, n)][m] for W, n, m in wanted])
            self._brdf_sets = wanted
        index = {k: j for j, k in enumerate(self._brdf_sets)}
        K = int(modes.max()) + 1
        beams = np.zeros((S, 2, M - 1))
        for s, sc in enumerate(self.scenarios):
            beams[s, 0] = glint_beam(M, self.mu, sc, K)[modes[s]]
        weights = np.zeros((S, 2))
        weights[:, 0] = 1.0
        eng.set_brdf_scenarios(np.array([index[k] for k in keys]), weights, beams)

    def _prepare(self, scenarios, order_caps=None):
        """Host side of a batch: tau profiles, per-scenario scalars, the table of distinct solar phase vectors with the rows
        and weights each scenario's first-order coefficients are made of (assembled on the device); phase functions met for the
        first time are appended to self._mats (the caller registers them)."""
        check_brdf(scenarios)
        self.scenarios = list(scenarios)
        L, M = self.L, self.M
        S = len(scenarios)
        # batch-sized host buffers are kept between batches (BatchSolver.update): fresh ones cost page faults every time
        bufs = getattr(self, "_host_bufs", None)
        if bufs is None or bufs[0].shape != (S, L):
            bufs = self._host_bufs = (np.empty((S, L)), np.arange(L, dtype=np.float64), np.arange(L))
        tau, rows_f, rows = bufs
        # tau profiles of the whole batch at once: the same arithmetic as grid.tau_profile, element for element
        # (the group key fixes idx_up / idx_down for every scenario of the batch; int -> float conversion is exact)
        t_atm = np.array([sc.tauStar_atm for sc in scenarios], dtype=np.float64)
        t_aer = np.array([sc.tauStar_aer for sc in scenarios], dtype=np.float64)
        iu, idn = self.idx_up, self.idx_down
        np.multiply(rows_f[None, :], t_atm[:, None], out=tau)
        np.divide(tau, L - 1, out=tau)
        tau[:, iu:idn + 1] += (rows[iu:idn + 1] + 1 - iu)[None, :] * (t_aer / (idn + 1 - iu))[:, None]
        tau[:, idn + 1:] += t_aer[:, None]
        self._new_mats = 0
        # phase tables: one look-up per DISTINCT (phase, mu0) of the batch; a scenario refers to rows of the table
        tab_rows = []
        hits = []          # (table row, operand index) of atmosphere and aerosol, scenario after scenario
        seen = {}
        for sc in scenarios:
            mu0 = sc.mu0
            for spec in (sc.atm_phase, sc.aer_phase):
                key = (spec if isinstance(spec[0], str) else id(spec[1]), mu0)
                hit = seen.get(key)
                if hit is None:
                    P0, P, k = self._phases.get(spec, M, self.mu, mu0, need_P=not self._device_phase)
                    if k not in self._mat_index:
                        self._mat_index[k] = len(self._mats)
                        self._mats.append(P)
                        self._mat_keys.append(k if k[0] != "array" else None)  # analytic families are immutable: cache on device
                        self._new_mats += 1
                    hit = seen[key] = (len(tab_rows), self._mat_index[k])
                    tab_rows.append(P0)
                hits.append(hit)
        both = np.array(hits, dtype=np.int32).reshape(S, 2, 2)
        p0_idx, mat_idx = np.ascontiguousarray(both[:, :, 0]), both[:, :, 1]
        tab = getattr(self, "_tab_buf", None)
        if tab is None or tab.shape[0] < len(tab_rows):
            tab = self._tab_buf = np.empty((max(len(tab_rows), 16), self.N))
        for r, P0 in enumerate(tab_rows):
            tab[r] = P0
        alb_atm = np.array([sc.alb_atm for sc in scenarios], dtype=np.float64)
        alb_aer = np.array([sc.alb_aer for sc in scenarios], dtype=np.float64)
        # global mixing weights (SOS_Aer_main_specular.py:52-53; note dtau_atm = tauStar_atm / L, Q9)
        dtau_aer = t_aer / (idn + 1 - iu)
        dtau_atm = t_atm / L
        f_atm = dtau_atm / (dtau_atm + dtau_aer)
        f_aer = dtau_aer / (dtau_atm + dtau_aer)
        # first-order coefficient planes C0 = P0_atm * alb_atm, C1 = C0 * f_atm + (P0_aer * alb_aer) * f_aer: the device assembles
        # them from the table (sos_first_order_tab, same operations in the same order); Ccoef does it on the host when asked
        self.P0tab = tab[: len(tab_rows)]
        self.P0idx = p0_idx
        self.P0w = np.stack([alb_atm, f_atm, alb_aer, f_aer], axis=1)
        coefs = np.zeros(S, dtype=_lib.SCENARIO_DTYPE)
        coefs["mu0"] = [sc.mu0 for sc in scenarios]
        coefs["grd_alb"] = [sc.grd_alb for sc in scenarios]
        coefs["tauStar_tot"] = t_atm + t_aer
        coefs["coef_atm"] = alb_atm
        coefs["coef_mix_atm"] = alb_atm * f_atm
        coefs["coef_mix_aer"] = alb_aer * f_aer
        coefs["threshold"] = [sc.threshold for sc in scenarios]
        coefs["phase_atm"] = mat_idx[:, 0]
        coefs["phase_aer"] = mat_idx[:, 1]
        coefs["extrap_width"][:, 0] = G.extrapolation_widths(tau[:, iu - 1], M)
        coefs["extrap_width"][:, 1] = coefs["extrap_width"][:, 2] = G.extrapolation_widths(tau[:, idn], M)
        if order_caps is not None:
            coefs["order_cap"] = order_caps
        self.tau = tau
        return coefs

    @property
    def Ccoef(self) -> np.ndarray:
        """The (S, 2, N) first-order coefficient planes of the batch, assembled on the host (sos_first_order's input)."""
        w = self.P0w
        C = np.empty((len(self.scenarios), 2, self.N))
        np.multiply(self.P0tab[self.P0idx[:, 0]], w[:, 0:1], out=C[:, 0])
        np.multiply(C[:, 0], w[:, 1:2], out=C[:, 1])
        C[:, 1] += (self.P0tab[self.P0idx[:, 1]] * w[:, 2:3]) * w[:, 3:4]
        return C

    def _register_phases(self):
        mats = list(self._mats)
        if self._device_phase:
            # analytic families: the N x N matrix is built on the device (sos_build_phase) unless its
            # contraction operand is already resident; only the cheap P0 vectors were built on the host
            for i, k in enumerate(self._mat_keys):
                if k is not None and mats[i] is None:
                    mats[i] = _DeviceBuilt(self.engine, k[0], k[1], tuple(k[3:5]) if len(k) > 3 else None)
        self.engine.set_phase(mats, keys=self._mat_keys)

    def update(self, scenarios: Sequence[Scenario], order_caps: Optional[Sequence[int]] = None,
               brdf_modes: Optional[Sequence[int]] = None):
        """Feed the solver its next batch (same grid group, same number of scenarios): the plan, its device buffers and
        the registered phase operands are kept (sos_plan_update); only tau, the per-scenario scalars and the first-order
        coefficients change.  What a parameter sweep calls between batches instead of building a new BatchSolver."""
        if len(scenarios) != len(self.scenarios) or {_group_key(s) for s in scenarios} != {self._key}:
            raise ValueError("BatchSolver.update: the next batch must keep the grid group and the batch size")
        coefs = self._prepare(scenarios, order_caps)
        if self._new_mats:
            if len(self._mats) > 16:
                raise ValueError("BatchSolver.update: more than 16 phase functions in one plan")
            self._register_phases()          # a phase function met for the first time: register the larger operand set
        self.engine.update(self.tau, coefs)
        if self._key[4] in ("rossli", "ocean"):
            self._send_brdf(brdf_modes)

    def first_order(self, also_into=None):
        if SosEngine.table_fits(self.P0tab.shape[0], len(self.scenarios), self.N):
            self.I1 = self.engine.first_order_from_table(self.P0tab, self.P0idx, self.P0w, out=self.I1, also_into=also_into)
        else:   # (a single scenario with two phase functions: nothing to save, the planes go up as they are)
            self.I1 = self.engine.first_order(self.Ccoef, out=self.I1, also_into=also_into)
        return self.I1

    def solve(self, keep_orders: int = 0, poll_every: int = 2, max_orders: Optional[int] = None):
        # the first-order kernel stores its values twice: into I1 and into the field the loop accumulates into (I = I_1 + ...),
        # which is one device-to-device field copy less per solve
        acc = self.engine._buf("I")
        I1 = self.first_order(also_into=acc)
        mo = max_orders if max_orders is not None else max(s.max_orders for s in self.scenarios)
        # the first order is recomputed by every solve, so its buffer can serve as the loop's I_n field -- unless the caller
        # wants the per-order fields back (results() then reads I1 as order 1)
        kw = dict(max_orders=mo, keep_orders=keep_orders, poll_every=poll_every, consume_I1=(keep_orders == 0), I=acc, I_holds_I1=True)
        try:
            return self.engine.solve(I1, **kw)
        except _lib.SosRetry:   # (see SosEngine.solve) -- the first order was consumed: rebuild it, the plan has switched kernels
            I1 = self.first_order(also_into=acc)
            return self.engine.solve(I1, **kw)

    def results(self, res, quadratures=True, keep_orders=0, fields=True) -> List[DriverResult]:
        """Per-scenario results on the host.  fields=False skips the D2H copy of the radiance fields
        (what a flux / forcing sweep needs: SOS_Aer_radiative_forcing returns one float)."""
        eng = self.engine
        I = eng.to_host(res.I).reshape(eng.S, eng.L, eng.N) if fields else None
        q = None
        if quadratures:
            q = eng.quadratures(res.I, self.z, direct_scale=1.0)
        orders = None
        if keep_orders and res.orders is not None:
            orders = res.orders[:, :, : eng.N].reshape(keep_orders, eng.S, eng.L, eng.N).cpu().numpy()
        I1 = eng.to_host(self.I1).reshape(eng.S, eng.L, eng.N) if (keep_orders and res.orders is not None) else None
        toa = None
        if q is not None:
            # TOA net flux with the F0/(4 pi) direct scaling (SOS_Aer_critical_albedo.py:377-382): same quadrature sums, direct
            # terms rescaled from F0 to F0/(4 pi) -- for the whole batch at once
            mu0 = np.array([sc.mu0 for sc in self.scenarios], dtype=np.float64)
            # (a diffuse Lambert, Ross-Li or ocean ground reflects the beam into the field: no collimated reflected term)
            alb = np.array([0.0 if sc.surface in DIFFUSE_GROUNDS else sc.grd_alb for sc in self.scenarios], dtype=np.float64)
            k = (np.pi / mu0) * (1.0 - 1.0 / (4 * np.pi))
            t0, tl = self.tau[:, 0], self.tau[:, -1]
            fd = q["flux_down"][:, 0] + k * np.exp(-t0 / mu0)
            fu = q["flux_up"][:, 0] - k * alb * np.exp(-(2 * tl - t0) / mu0)
            toa = -fd - fu
        tau_out = self.tau.copy()   # (self.tau is a buffer reused by the next update())
        if np.any(res.status & _lib.STATUS_BLEND_OVERRUN):
            raise IndexError("mu->0 blend search ran off the row (reference: IndexError, "
                             "SOS_Aer_main_specular.py:404)")
        # per-scenario records: NumPy scalars and rows are unpacked once for the whole batch (a sweep calls this per batch)
        n_l = [int(v) for v in res.n_orders]
        ratio_l = np.maximum(res.ratio_toa, res.ratio_surf).tolist()
        status_l = res.status.tolist()
        tau_l = list(tau_out)
        I_l = list(I) if fields else [None] * len(n_l)
        if q is not None:
            fu, fd, nf, df = list(q["flux_up"]), list(q["flux_down"]), list(q["net_flux"]), list(q["diffusivity"])
            hr = list(q["heating_rate"]) if q["heating_rate"] is not None else [None] * len(n_l)
            toa_l = toa.tolist()
        out = []
        for i in range(len(self.scenarios)):
            r = DriverResult(I=I_l[i], n=n_l[i], tau=tau_l[i], mu=self.mu, z_profile=self.z, idx_up=self.idx_up,
                             idx_down=self.idx_down, ratio=ratio_l[i], status=status_l[i])
            if q is not None:
                r.flux_up, r.flux_down, r.net_flux, r.diffusivity, r.heating_rate = fu[i], fd[i], nf[i], df[i], hr[i]
                r.toa_net_flux = toa_l[i]
            if orders is not None:
                r.I_saved = [I1[i]] + [orders[k, i] for k in range(min(keep_orders, r.n - 1))]
            out.append(r)
        return out


MAX_PHASES_PER_PLAN, MAX_GROUPS_PER_PLAN = 16, 48   # SOS_MAX_PHASE / SOS_MAX_GROUPS of the C ABI (csrc/common.cuh)


def _phase_id(spec):
    return spec if isinstance(spec[0], str) else ("array", id(spec[1]))


def split_for_plan_limits(scenarios: Sequence[Scenario], idxs: Sequence[int], max_phases: int = MAX_PHASES_PER_PLAN,
                          brdf_modes: Optional[Sequence[int]] = None) -> List[List[int]]:
    """Cut one grid group into sub-batches a plan accepts: at most 16 (max_phases) distinct phase matrices, 48 (atm, aer)
    operand pairs and 64 ocean glint sets (distinct (wind_speed, ocean_index, mode); brdf_modes: the mode of every scenario,
    None = 0) each (a phase sweep over more than 16 HG asymmetry factors, per-scenario Mie arrays or a wind-speed sweep would
    otherwise be refused by the plan).  Order inside the group is kept."""
    out, cur, phases, pairs, sets = [], [], set(), set(), set()
    for i in idxs:
        sc = scenarios[i]
        pa, pe = _phase_id(sc.atm_phase), _phase_id(sc.aer_phase)
        gs = {_glint_key(sc, brdf_modes[i] if brdf_modes is not None else 0)} if sc.surface == "ocean" else set()
        new_phases = phases | {pa, pe}
        new_pairs = pairs | {(pa, pe), (pa, None)}
        new_sets = sets | gs
        if cur and (len(new_phases) > max_phases or len(new_pairs) > MAX_GROUPS_PER_PLAN or len(new_sets) > MAX_BRDF_SETS_PER_PLAN):
            out.append(cur)
            cur, new_phases, new_pairs, new_sets = [], {pa, pe}, {(pa, pe), (pa, None)}, gs
        cur.append(i)
        phases, pairs, sets = new_phases, new_pairs, new_sets
    if cur:
        out.append(cur)
    return out


def solve_scenarios(scenarios: Sequence[Scenario], device=None, keep_orders: int = 0, quadratures: bool = True,
                    fold: Optional[bool] = None) -> List[DriverResult]:
    """Solve any mix of scenarios; those sharing a grid are batched together.  fold: see SosEngine."""
    out: List[Optional[DriverResult]] = [None] * len(scenarios)
    for idxs, _, _, results in solved_batches(scenarios, device=device, keep_orders=keep_orders, quadratures=quadratures,
                                              fold=fold):
        for i, r in zip(idxs, results):
            out[i] = r
    return out  # type: ignore


def grid_groups(scenarios: Sequence[Scenario]) -> List[List[int]]:
    """Indices of the scenarios that share a grid (layers, angles, aerosol rows, surface), group by group."""
    groups: Dict[tuple, List[int]] = {}
    for i, sc in enumerate(scenarios):
        groups.setdefault(_group_key(sc), []).append(i)
    return list(groups.values())


def solved_batches(scenarios: Sequence[Scenario], device=None, keep_orders: int = 0, quadratures: bool = True,
                   fold: Optional[bool] = None, groups: Optional[List[List[int]]] = None):
    """The batches of solve_scenarios one at a time: yields (indices, BatchSolver, SolveResult, [DriverResult]) while the
    batch's plan and device fields are still alive (the plan is closed when the caller asks for the next batch)."""
    check_brdf(scenarios)   # (before the first batch touches the device)
    groups = grid_groups(scenarios) if groups is None else groups
    for idxs in [b for g in groups for b in split_for_plan_limits(scenarios, g)]:
        bs = BatchSolver([scenarios[i] for i in idxs], device=device, fold=fold)
        try:
            res = bs.solve(keep_orders=keep_orders)
            yield idxs, bs, res, bs.results(res, quadratures=quadratures, keep_orders=keep_orders)
        finally:
            bs.engine.close()


def SOS_Aer_main_specular(keep_orders: int = 0, device=None, **params) -> DriverResult:
    """SOS_Aer() of SOS_Aer_main_specular.py with keyword parameters; returns the arrays."""
    sc = Scenario(**dict(params, surface="specular"))
    return solve_scenarios([sc], device=device, keep_orders=keep_orders)[0]


def SOS_Aer_main_lambertian(keep_orders: int = 0, device=None, **params) -> DriverResult:
    """SOS_Aer() of SOS_Aer_main_lambertian.py (Lambert-as-coded, first order as in the specular driver)."""
    sc = Scenario(**dict(params, surface="lambert"))
    return solve_scenarios([sc], device=device, keep_orders=keep_orders)[0]


def SOS_Aer_radiative_forcing(tauStar_aer, dtau_aer, tauStar_atm, dtau_atm, P_aer, P0_aer, alb_aer, P_atm, P0_atm,
                              alb_atm, grd_alb, F0, mu, mu0, nb_angles, tau, nb_layers, idx_up, idx_down,
                              tauStar_tot=None, baseline="reference", device=None):
    """Drop-in for SOS_Aer_critical_albedo.py:20 (19 positional arguments).

    The reference reads `tauStar_tot` from a module global (:39) -- pass it as a keyword (default:
    tau[-1]).  Its baseline recursion (:385-389) reuses the same tau/dtau/P/omega, so the returned
    forcing is identically 0 (Q19); baseline="reference" reproduces that, baseline="none" returns the
    TOA net flux of this single solve (the quantity a corrected sweep needs).
    """
    tau = np.ascontiguousarray(tau, dtype=np.float64)
    mu = np.ascontiguousarray(mu, dtype=np.float64)
    M, L = int(nb_angles), int(nb_layers)
    T = float(tauStar_tot) if tauStar_tot is not None else float(tau[-1])
    f_atm = dtau_atm / (dtau_atm + dtau_aer)
    f_aer = dtau_aer / (dtau_atm + dtau_aer)
    widths = (G.extrapolation_width(float(tau[idx_up - 1]), M), G.extrapolation_width(float(tau[idx_down]), M),
              G.extrapolation_width(float(tau[idx_down]), M))
    coef = ScenarioCoefficients(mu0=float(mu0), grd_alb=float(grd_alb), tauStar_tot=T, coef_atm=float(alb_atm),
                                coef_mix_atm=float(alb_atm * f_atm), coef_mix_aer=float(alb_aer * f_aer),
                                phase_atm=0, phase_aer=1, extrap_width=widths)
    eng = SosEngine(mu, tau[None, :], [coef], [0, int(idx_up), int(idx_down) + 1, L], _lib.SURFACE_SPECULAR, device=device)
    try:
        eng.set_phase([P_atm, P_aer])
        Cc = np.empty((1, 2, 2 * M))
        Cc[0, 0] = alb_atm * np.asarray(P0_atm)
        Cc[0, 1] = alb_atm * np.asarray(P0_atm) * f_atm + alb_aer * np.asarray(P0_aer) * f_aer
        I1 = eng.first_order(Cc)
        res = eng.solve(I1)
        q = eng.quadratures(res.I, None, direct_scale=1.0 / (4 * np.pi), heating=False)
        # the kernels use F0 = pi/mu0 (SOS_Aer_main_specular.py:105); the solve is linear in F0
        net = float(-q["flux_down"][0][0] - q["flux_up"][0][0]) * (float(F0) * float(mu0) / np.pi)
    finally:
        eng.close()
    if tauStar_aer == 0 or baseline == "none":
        return net
    return net - net  # the reference's recursion recomputes the identical solve (Q19)


def SOS_Aer_critical_albedo(tauStar_aer, dtau_aer, tauStar_atm, dtau_atm, P_aer, P0_aer, P_atm, P0_atm, alb_atm, grd_alb,
                            F0, mu, mu0, nb_angles, tau, nb_layers, idx_up, idx_down, tauStar_tot=None, device=None):
    """Drop-in for SOS_Aer_critical_albedo.py:394-410: bisection on the aerosol single-scattering albedo.

    As shipped the forcing it bisects on is identically zero (its baseline recursion repeats the same
    solve, Q19), so the first tested value 0.5 is returned after one solve; that behaviour is reproduced.
    `critical_albedo_sweep` below is the corrected, batched version.
    """
    lo, hi = 0.0, 1.0
    while (hi - lo) > 0.1:
        mid = (hi + lo) / 2
        f = SOS_Aer_radiative_forcing(tauStar_aer, dtau_aer, tauStar_atm, dtau_atm, P_aer, P0_aer, mid, P_atm, P0_atm,
                                      alb_atm, grd_alb, F0, mu, mu0, nb_angles, tau, nb_layers, idx_up, idx_down,
                                      tauStar_tot=tauStar_tot, baseline="reference", device=device)
        if abs(f) < 0.001:
            return mid
        if f > 0:
            lo = mid
        else:
            hi = mid
    return (hi + lo) / 2


def critical_albedo_sweep(points: Sequence[Scenario], width: float = 0.1, forcing_tol: float = 1e-3, device=None,
                          max_iter: int = 20, return_evaluated: bool = False):
    """Critical aerosol single-scattering albedo for many sweep points at once (config 5's real caller).

    For every point (a Scenario; its alb_aer is ignored) bisect omega_aer in [0, 1] on the radiative
    forcing  dF = F_net_TOA(tau_aer, omega) - F_net_TOA(tau_aer = 0)  with a GENUINE aerosol-free
    baseline (documented deviation from SOS_Aer_critical_albedo.py:385-389, whose baseline repeats the
    same solve).  Stopping rule as in :397,402: interval width <= `width` or |dF| < `forcing_tol`.
    Every bisection step is ONE batched GPU solve over all still-open points.
    Returns (omega_critical, forcing, n_solves): `forcing[i]` is the forcing at the LAST omega solved for point i;
    that omega is returned as a fourth array with return_evaluated=True (omega_critical is the same value when the sweep
    stopped on |dF| < forcing_tol, otherwise the midpoint of the final bracket, at most width/2 away).
    """
    pts = list(points)
    base = solve_scenarios([replace(p, tauStar_aer=0.0, alb_aer=1.0) for p in pts], device=device)
    f0 = np.array([r.toa_net_flux for r in base])
    lo = np.zeros(len(pts))
    hi = np.ones(len(pts))
    omega = np.full(len(pts), 0.5)
    forcing = np.full(len(pts), np.nan)
    open_ = np.ones(len(pts), dtype=bool)
    n_solves = len(pts)
    for _ in range(max_iter):
        open_ &= (hi - lo) > width
        idx = np.nonzero(open_)[0]
        if idx.size == 0:
            break
        mid = (hi[idx] + lo[idx]) / 2
        res = solve_scenarios([replace(pts[i], alb_aer=float(m)) for i, m in zip(idx, mid)], device=device)
        n_solves += idx.size
        f = np.array([r.toa_net_flux for r in res]) - f0[idx]
        omega[idx], forcing[idx] = mid, f
        close = np.abs(f) < forcing_tol
        open_[idx[close]] = False
        up = (f > 0) & ~close
        lo[idx[up]] = mid[up]
        hi[idx[~up & ~close]] = mid[~up & ~close]
    still = (hi - lo) <= width
    final = np.where(np.isnan(forcing) | (still & (np.abs(np.nan_to_num(forcing)) >= forcing_tol)), (hi + lo) / 2, omega)
    if return_evaluated:
        return final, forcing, n_solves, omega
    return final, forcing, n_solves
