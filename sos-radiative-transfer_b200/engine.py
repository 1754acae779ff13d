"""SosEngine: a batch of scenarios sharing one (layers x mu) grid, resident on one B200.

Thin host object over the C ABI (include/sos_b200.h): it owns the torch device buffers
(PyTorch is used for device memory and streams only), precomputes the once-per-grid tables
(mu weights, chunking, extrapolation matrices) and exposes the per-order operators of the
reference -- first order, source contraction, layer sweeps, accumulate/convergence -- plus the
whole order loop and the quadratures.  No CPU fallback: every method raises if the CUDA
library is missing.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from . import grid as G


def _align(n: int, a: int) -> int:
    return (n + a - 1) // a * a


_PINNED = {}
_OPERANDS = {}  # device-resident contraction operands shared between engines (see SosEngine.set_phase)
_FOLDED = {}    # their folded counterparts [B+ | B-] and centrosymmetry defects (sos_build_folded)
FOLD_DEFECT_MAX = 1e-12  # fold only operands that are centrosymmetric to rounding (observed <= 3e-14 for every builder)
_LOWRANK = {}   # low-rank factors (Ut, Vt, rank) of the operands, see SosEngine._lowrank_factors
LOWRANK_RESIDUAL_MAX = 1e-14   # accept the closed-form factors only if max|A - Ut^T Vt| <= this * max|A| (observed ~2e-16)


def _pinned_pair(elems: int):
    """Two grow-only pinned float64 staging buffers shared by all engines of the process."""
    have = _PINNED.get("pair")
    if have is None or have[0].numel() < elems:
        have = [torch.empty(elems, dtype=torch.float64, pin_memory=True) for _ in range(2)]
        _PINNED["pair"] = have
    return have


@dataclass
class ScenarioCoefficients:
    """Per-scenario scalars in the units the kernels want (see sos_scenario in sos_b200.h)."""
    mu0: float
    grd_alb: float
    tauStar_tot: float
    coef_atm: float
    coef_mix_atm: float = 0.0
    coef_mix_aer: float = 0.0
    threshold: float = 1e-4
    phase_atm: int = 0
    phase_aer: int = 0
    extrap_width: Sequence[int] = (0, 0, 0)
    order_cap: int = 0   # > 0: sum exactly orders 1 .. order_cap, ignoring the threshold (an azimuthal mode m >= 1)


class SolveResult:
    """What the order loop returns: accumulated field + per-scenario bookkeeping."""

    def __init__(self, I, n_orders, ratio_toa, ratio_surf, status, orders=None, active=None):
        self.I = I
        self.active = active      # 1 where the loop stopped at max_orders before the scenario converged (status bit MAX_ORDERS)
        self.n_orders = n_orders
        self.ratio_toa = ratio_toa
        self.ratio_surf = ratio_surf
        self.status = status
        self.orders = orders


class SosEngine:
    def __init__(self, mu, tau, scenarios: Sequence[ScenarioCoefficients], region_start: Sequence[int],
                 surface: int, device: Optional[torch.device] = None, chunk_rows: int = 0, fold: Optional[bool] = None):
        """fold: use the folded contraction (half the multiply-adds) when every operand is centrosymmetric;
        None = on unless the environment says SOS_B200_FOLD=0."""
        self.lib = _lib.load()
        self.fold = (os.environ.get("SOS_B200_FOLD", "1") != "0") if fold is None else bool(fold)
        self.folded = False
        self.lowrank = []         # numerical rank per operand (0 = dense), set by set_phase in fold mode
        self.fold_defect = None   # centrosymmetry defect of the operands (set by set_phase when the fold is considered)
        if not torch.cuda.is_available():
            raise _lib.SosError("no CUDA device: the SOS engine has no CPU fallback")
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        mu = np.ascontiguousarray(mu, dtype=np.float64)
        tau = np.ascontiguousarray(np.atleast_2d(tau), dtype=np.float64)
        self.N = mu.shape[0]
        self.M = self.N // 2
        self.S, self.L = tau.shape
        if len(scenarios) != self.S:
            raise ValueError("one ScenarioCoefficients per tau row expected")
        self.mu, self.tau = mu, tau
        self.ld = _align(self.N, 16)  # 128-byte rows: TMA boxes of the contraction stay line-aligned
        self.n_regions = len(region_start) - 1
        self.region_start = list(region_start)
        self.surface = surface
        self.scenarios = scenarios

        g = _lib.sos_grid()
        g.nb_layers, g.nb_angles, g.n_scenarios, g.n_regions = self.L, self.M, self.S, self.n_regions
        for i in range(4):
            g.region_start[i] = self.region_start[i] if i < len(self.region_start) else 0
        g.surface, g.ld, g.chunk_rows = surface, self.ld, chunk_rows
        W = np.ascontiguousarray(G.extrapolation_tables(mu, self.M), dtype=np.float64)
        self._plan = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_plan_create(C.byref(self._plan), C.byref(g), mu.ctypes.data, tau.ctypes.data,
                                                self._scenario_array(scenarios), W.ctypes.data if W.size else None, int(W.size)),
                       "sos_plan_create")
        self._A = []          # device contraction matrices (keep alive)
        self._bufs = {}

    def _scenario_array(self, scenarios):
        """ctypes view of the per-scenario records: a list of ScenarioCoefficients, or a NumPy record array of
        _lib.SCENARIO_DTYPE (what BatchSolver builds for a whole batch at once)."""
        if isinstance(scenarios, np.ndarray):
            if scenarios.dtype != _lib.SCENARIO_DTYPE or scenarios.shape != (self.S,):
                raise ValueError("scenario table: expected %d records of _lib.SCENARIO_DTYPE" % self.S)
            self._scen_keepalive = np.ascontiguousarray(scenarios)
            return C.cast(self._scen_keepalive.ctypes.data, C.POINTER(_lib.sos_scenario))
        sc = (_lib.sos_scenario * self.S)()
        for i, s in enumerate(scenarios):
            sc[i].mu0, sc[i].grd_alb, sc[i].tauStar_tot = s.mu0, s.grd_alb, s.tauStar_tot
            sc[i].coef_atm, sc[i].coef_mix_atm, sc[i].coef_mix_aer = s.coef_atm, s.coef_mix_atm, s.coef_mix_aer
            sc[i].threshold = s.threshold
            sc[i].phase_atm, sc[i].phase_aer = s.phase_atm, s.phase_aer
            for k in range(3):
                sc[i].extrap_width[k] = int(s.extrap_width[k]) if k < len(s.extrap_width) else 0
            sc[i].order_cap = int(s.order_cap)
        return sc

    def update(self, tau, scenarios: Sequence[ScenarioCoefficients]):
        """The next batch on the same grid (sos_plan_update): new tau profiles and per-scenario scalars, same phase
        matrices; device buffers, tensor maps and operands are kept."""
        tau = np.ascontiguousarray(np.atleast_2d(tau), dtype=np.float64)
        if tau.shape != (self.S, self.L) or len(scenarios) != self.S:
            raise ValueError("update: the batch must keep its shape (S scenarios x L layers)")
        n = len(self._A)
        if isinstance(scenarios, np.ndarray):
            bad = bool(np.any(scenarios["phase_atm"] >= n) or np.any(scenarios["phase_aer"] >= n))
        else:
            bad = any(s.phase_atm >= n or s.phase_aer >= n for s in scenarios)
        if bad:
            raise ValueError("update: scenario refers to a phase matrix that is not registered")
        self.tau, self.scenarios = tau, scenarios
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_plan_update(self._plan, tau.ctypes.data, self._scenario_array(scenarios), self._stream),
                       "sos_plan_update")

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_plan", None) is not None and self._plan.value:
            with torch.cuda.device(self.device):   # (the library also switches to the plan's device itself)
                self.lib.sos_plan_destroy(self._plan)
            self._plan = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def new_field(self, zero=False):
        f = torch.zeros if zero else torch.empty
        return f((self.S * self.L, self.ld), dtype=torch.float64, device=self.device)

    def _buf(self, name):
        if name not in self._bufs:
            self._bufs[name] = self.new_field(zero=True)
        return self._bufs[name]

    def to_field(self, arr) -> torch.Tensor:
        """Host (S, L, N) / (L, N) array (or device tensor) -> padded device field."""
        if isinstance(arr, torch.Tensor) and arr.is_cuda and arr.shape == (self.S * self.L, self.ld):
            return arr
        a = torch.as_tensor(np.ascontiguousarray(arr, dtype=np.float64)) if not isinstance(arr, torch.Tensor) else arr
        a = a.reshape(self.S * self.L, self.N)
        out = self.new_field(zero=True)
        out[:, : self.N].copy_(a, non_blocking=False)
        return out

    def to_host(self, field: torch.Tensor) -> np.ndarray:
        """Device field -> fresh C-contiguous float64 (S, L, N) NumPy array ((L, N) when S == 1).

        Goes through two cached pinned staging buffers so that the PCIe copy of chunk k+1 overlaps the
        host memcpy of chunk k (a pageable .cpu() of a large field runs at ~2 GB/s).
        """
        rows = self.S * self.L
        out = np.empty((rows, self.N), dtype=np.float64)
        chunk = max(1, min(rows, (32 << 20) // (8 * self.N)))
        stage = _pinned_pair(chunk * self.N)
        stream = torch.cuda.current_stream(self.device)
        events = [torch.cuda.Event(), torch.cuda.Event()]
        pending = []
        with torch.cuda.device(self.device):
            for k, r0 in enumerate(range(0, rows, chunk)):
                r1 = min(rows, r0 + chunk)
                buf = stage[k & 1][: (r1 - r0) * self.N].view(r1 - r0, self.N)
                if len(pending) == 2:  # this buffer's previous contents must be consumed first
                    pr0, pr1, pbuf, pev = pending.pop(0)
                    pev.synchronize()
                    out[pr0:pr1] = pbuf.numpy()
                buf.copy_(field[r0:r1, : self.N], non_blocking=True)
                events[k & 1] = torch.cuda.Event()
                events[k & 1].record(stream)
                pending.append((r0, r1, buf, events[k & 1]))
            for pr0, pr1, pbuf, pev in pending:
                pev.synchronize()
                out[pr0:pr1] = pbuf.numpy()
        a = out.reshape(self.S, self.L, self.N)
        return a[0] if self.S == 1 else a

    @property
    def gensrc_enabled(self) -> bool:
        """True when sos_solve may rebuild sources inside the sweeps on this plan (SOS_B200_GENSRC=0 disables it; a blend
        wider than the columns kept raw disables it for the plan at run time)."""
        return bool(self.lib.sos_plan_query(self._plan, _lib.QUERY_FUSED_ORDER) == 1)

    @property
    def generated_source(self) -> bool:
        """True when sos_solve rebuilds J on the molecular rows from two projections per row instead of writing and reading
        it (csrc/sweep.cuh: SrcGen): needs the folded contraction and rank <= 2 molecular operands."""
        return bool(self.lib.sos_plan_query(self._plan, _lib.QUERY_GENERATED_SOURCE) == 1)

    @property
    def launches(self) -> int:
        return int(self.lib.sos_launch_count(self._plan))

    # ------------------------------------------------------------------ phase operands
    def set_phase(self, matrices: Sequence, keys: Optional[Sequence] = None):
        """Upload the phase matrices P (N, N) once and build A[k,m] = w_k/4 P[m, N-1-k] on device.

        keys: optional hashable identity per matrix (e.g. ("hg", 0.5, M)); operands built for a key are
        kept on the device and shared by later engines of the same grid ("uploaded once", north_star).
        Only pass keys for matrices that are never modified in place."""
        self._A = []
        lda = self.ld
        self.h2d_phase_bytes = 0
        cks = []
        with torch.cuda.device(self.device):
            for i, P in enumerate(matrices):
                ck = None
                if keys is not None and keys[i] is not None:
                    ck = (keys[i], self.device.index, self.N, lda, self.mu.tobytes())
                    hit = _OPERANDS.get(ck)
                    if hit is not None:
                        self._A.append(hit)
                        cks.append(ck)
                        continue
                cks.append(ck)
                if hasattr(P, "build"):
                    Pd = P.build()            # built on the device (drivers._DeviceBuilt)
                elif isinstance(P, torch.Tensor):
                    Pd = P.to(self.device, torch.float64).contiguous()
                else:
                    Pd = torch.as_tensor(np.ascontiguousarray(P, dtype=np.float64)).to(self.device)
                    self.h2d_phase_bytes += Pd.numel() * 8
                if Pd.shape != (self.N, self.N):
                    raise ValueError(f"phase matrix must be ({self.N}, {self.N})")
                A = torch.zeros((self.N, lda), dtype=torch.float64, device=self.device)
                _lib.check(self.lib.sos_build_contraction(self._plan, Pd.data_ptr(), self.N, A.data_ptr(), lda, self._stream),
                           "sos_build_contraction")
                torch.cuda.current_stream(self.device).synchronize()  # Pd may be freed after this
                if ck is not None:
                    if len(_OPERANDS) >= 32:   # bounded: ~8 MB per operand at N = 1002
                        _OPERANDS.pop(next(iter(_OPERANDS)))
                    _OPERANDS[ck] = A
                self._A.append(A)
            ptrs = (C.c_void_p * len(self._A))(*[a.data_ptr() for a in self._A])
            _lib.check(self.lib.sos_plan_set_phase(self._plan, ptrs, len(self._A), lda), "sos_plan_set_phase")
            self.folded = False
            if self.fold:
                self._set_folded(cks)

    def _set_folded(self, cks):
        """Build (or fetch) the folded operand of every contraction matrix; enable the folded kernel when all
        of them are centrosymmetric to rounding (sos_b200.h: sos_build_folded / sos_plan_set_folded)."""
        rows, ldf = C.c_int(), C.c_int()
        self.lib.sos_fold_layout(self.M, C.byref(rows), C.byref(ldf))
        self._F, self.fold_defect = [], 0.0
        for A, ck in zip(self._A, cks):
            hit = _FOLDED.get(ck) if ck is not None else None
            if hit is None:
                F = torch.empty((rows.value, ldf.value), dtype=torch.float64, device=self.device)
                defect = C.c_double()
                _lib.check(self.lib.sos_build_folded(self._plan, A.data_ptr(), self.ld, F.data_ptr(), ldf.value,
                                                     C.byref(defect), self._stream), "sos_build_folded")
                hit = (F, defect.value)
                if ck is not None:
                    if len(_FOLDED) >= 32:
                        _FOLDED.pop(next(iter(_FOLDED)))
                    _FOLDED[ck] = hit
            self._F.append(hit[0])
            self.fold_defect = max(self.fold_defect, hit[1])
        if self.fold_defect <= FOLD_DEFECT_MAX:
            self._set_lowrank(cks)
            ptrs = (C.c_void_p * len(self._F))(*[f.data_ptr() for f in self._F])
            _lib.check(self.lib.sos_plan_set_folded(self._plan, ptrs, len(self._F), ldf.value), "sos_plan_set_folded")
            self.folded = True

    def _lowrank_factors(self, A: torch.Tensor):
        """(Ut, Vt, rank) with A = (Ut^T)(Vt) to rounding, or (None, None, 0).

        No SVD: every row of a Rayleigh / isotropic operand is affine in mu_m^2 (csrc/gemm_lowrank.cuh), so the factors are
        read off two columns of the operand on the device (sos_build_lowrank_mu2) and accepted only when they reproduce the
        dense operand to LOWRANK_RESIDUAL_MAX of its largest entry; every other operand stays dense."""
        rows, ldr = C.c_int(), C.c_int()
        self.lib.sos_lowrank_layout(self.M, C.byref(rows), C.byref(ldr))
        Ut = torch.empty((rows.value, ldr.value), dtype=torch.float64, device=self.device)
        Vt = torch.empty((rows.value, ldr.value), dtype=torch.float64, device=self.device)
        resid, rank = C.c_double(), C.c_int()
        _lib.check(self.lib.sos_build_lowrank_mu2(self._plan, A.data_ptr(), self.ld, Ut.data_ptr(), Vt.data_ptr(), ldr.value,
                                                  C.byref(resid), C.byref(rank), self._stream), "sos_build_lowrank_mu2")
        if not (resid.value <= LOWRANK_RESIDUAL_MAX):
            return None, None, 0
        return Ut, Vt, int(rank.value)

    def _set_lowrank(self, cks):
        """Register the low-rank factors of the operands that have them (sos_plan_set_lowrank); SOS_B200_LOWRANK=0 skips it."""
        n = len(self._A)
        self.lowrank = [0] * n
        if os.environ.get("SOS_B200_LOWRANK", "1") == "0":
            return
        self._LR = []
        for i, (A, ck) in enumerate(zip(self._A, cks)):
            hit = _LOWRANK.get(ck) if ck is not None else None
            if hit is None:
                hit = self._lowrank_factors(A)
                if ck is not None:
                    if len(_LOWRANK) >= 32:
                        _LOWRANK.pop(next(iter(_LOWRANK)))
                    _LOWRANK[ck] = hit
            self._LR.append(hit)
            self.lowrank[i] = hit[2]
        if not any(self.lowrank):
            return
        ut = (C.c_void_p * n)(*[(h[0].data_ptr() if h[2] else None) for h in self._LR])
        vt = (C.c_void_p * n)(*[(h[1].data_ptr() if h[2] else None) for h in self._LR])
        rk = (C.c_int * n)(*self.lowrank)
        ldr = next(h[0].shape[1] for h in self._LR if h[2])
        _lib.check(self.lib.sos_plan_set_lowrank(self._plan, ut, vt, rk, n, ldr), "sos_plan_set_lowrank")

    def build_phase_matrix(self, name: str, g: float = 0.5, mu0: Optional[float] = None):
        """P(mu, mu') (and P0(mu, mu0) when mu0 is given) of an analytic family, built ON THE DEVICE
        (sos_build_phase): 'rayleigh', 'hg', 'fwc', 'mie_lognormal' (g = (wl, n_re, n_im, r_m, sigma)), 'iso'.  Returns (P (N, N) tensor, P0 (N,) tensor or None)."""
        from . import phase as PH
        N = self.N
        P = torch.empty((N, N), dtype=torch.float64, device=self.device)
        P0 = torch.empty(N, dtype=torch.float64, device=self.device) if mu0 is not None else None
        if name == "iso":
            P.fill_(2.0)
            if P0 is not None:
                P0.fill_(1.0)
            return P, P0
        fam = {"rayleigh": 0, "hg": 1, "fwc": 2, "mie_lognormal": 2}[name]
        phi = np.linspace(0, np.pi, PH.NB_PHI)
        cphi = np.ascontiguousarray(np.cos(0 - phi))
        tx = ty = None
        tn = 0
        if fam == 2:
            # tabulated families: FWC cloud, or the log-normal Mie mixture of mie.py (g = its parameter tuple)
            key = ("phase_table", name, tuple(g) if isinstance(g, (tuple, list)) else None, self.device.index)
            if key not in _OPERANDS:
                xs, ys = PH.phase_table(name, g)
                _OPERANDS[key] = (torch.as_tensor(np.array(xs, dtype=np.float64)).to(self.device),
                                  torch.as_tensor(np.array(ys, dtype=np.float64)).to(self.device))
            tx, ty = _OPERANDS[key]
            tn = tx.numel()
        gval = float(g) if not isinstance(g, (tuple, list)) else 0.0
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_build_phase(self._plan, fam, gval, float(mu0 if mu0 is not None else 0.5),
                                                phi.ctypes.data, cphi.ctypes.data,
                                                tx.data_ptr() if tx is not None else None,
                                                ty.data_ptr() if ty is not None else None, int(tn),
                                                P.data_ptr(), N, P0.data_ptr() if P0 is not None else None, self._stream),
                       "sos_build_phase")
        return P, P0

    def build_phase_modes(self, name: str, g: float = 0.5, n_modes: int = 1, mu0: Optional[float] = None, n_quad: int = 25,
                          want_P: bool = True):
        """Azimuthal Fourier modes m = 0 .. n_modes-1 of a phase function, built ON THE DEVICE (sos_build_phase_modes) with
        n_quad azimuth nodes on [0, pi]: (P (n_modes, N, N) tensor or None, P0 (n_modes, N) tensor or None).  Families as in
        build_phase_matrix; every mode is normalised by the column integrals of mode 0 (phase.phase_modes is the NumPy
        reference).  At n_quad = 25 mode 0 is bit for bit build_phase_matrix."""
        from . import phase as PH
        N, K = self.N, int(n_modes)
        P = torch.empty((K, N, N), dtype=torch.float64, device=self.device) if want_P else None
        P0 = torch.empty((K, N), dtype=torch.float64, device=self.device) if mu0 is not None else None
        if name == "iso":
            for t, v in ((P, 2.0), (P0, 1.0)):
                if t is not None:
                    t.zero_()
                    t[0].fill_(v)
            return P, P0
        fam = {"rayleigh": 0, "hg": 1, "fwc": 2, "mie_lognormal": 2}[name]
        phi, cphi = PH.azimuth_nodes(n_quad, K)
        tx = ty = None
        if fam == 2:
            xs, ys = PH.phase_table(name, g)
            tx = torch.as_tensor(np.array(xs, dtype=np.float64)).to(self.device)
            ty = torch.as_tensor(np.array(ys, dtype=np.float64)).to(self.device)
        gval = float(g) if not isinstance(g, (tuple, list)) else 0.0
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_build_phase_modes(self._plan, fam, gval, float(mu0 if mu0 is not None else 0.5), int(n_quad),
                                                      phi.ctypes.data, cphi.ctypes.data, K,
                                                      tx.data_ptr() if tx is not None else None,
                                                      ty.data_ptr() if ty is not None else None, int(tx.numel()) if tx is not None else 0,
                                                      P.data_ptr() if P is not None else None, N, N * N,
                                                      P0.data_ptr() if P0 is not None else None, self._stream),
                       "sos_build_phase_modes")
            torch.cuda.current_stream(self.device).synchronize()   # (the table tensors may be freed after this)
        return P, P0

    # ------------------------------------------------------------------ Ross-Li ground
    def build_brdf_modes(self, n_modes: int = 1, n_quad: Optional[int] = None) -> torch.Tensor:
        """Fourier modes 0 .. n_modes-1 of the two Ross-Li kernels on this grid, built ON THE DEVICE (sos_build_brdf_modes):
        a (2, n_modes, M, ldr) tensor, [k][m][c][i] = rho_{k,m}(mu[M+1+i], |mu[c]|) for k = vol, geo (the transposed
        layout the coupling reads; ldr = M-1 rounded up to even).  brdf.brdf_modes is the NumPy reference ([m][i][c])."""
        from . import brdf as BR
        K, nq = int(n_modes), int(n_quad if n_quad is not None else BR.BRDF_NODES)
        M = self.M
        ldr = _align(M - 1, 2)
        R = torch.zeros((2, K, M, ldr), dtype=torch.float64, device=self.device)
        phi, tab = BR.node_table(nq, K)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_build_brdf_modes(self._plan, nq, phi.ctypes.data, tab.ctypes.data, K, BR.BRDF_MU_MIN,
                                                     R[0].data_ptr(), R[1].data_ptr(), ldr, M * ldr, self._stream),
                       "sos_build_brdf_modes")
            torch.cuda.current_stream(self.device).synchronize()   # (phi / tab are host temporaries)
        return R

    def set_brdf(self, pairs: Sequence):
        """Register the mode matrix sets of a Ross-Li or ocean plan (sos_plan_set_brdf): for Ross-Li pairs[j] = (vol, geo),
        two (M, ldr) device tensors in the layout of build_brdf_modes (e.g. R[0, m], R[1, m]); for the ocean pairs[j] = one
        (M, ldr) glint matrix of build_glint_modes (e.g. R[m]).  The engine keeps them alive."""
        if not len(pairs):
            raise ValueError("set_brdf: at least one mode matrix set")
        sets = [(p,) if isinstance(p, torch.Tensor) else tuple(p) for p in pairs]
        ldr = sets[0][0].shape[-1]
        for P in (t for st in sets for t in st):
            if P.shape != (self.M, ldr) or P.dtype != torch.float64 or not P.is_contiguous() or P.device != self.device:
                raise ValueError("set_brdf: every matrix must be a contiguous float64 (M, ldr) tensor on the plan's device")
        if len({len(st) for st in sets}) != 1:
            raise ValueError("set_brdf: every set has the same number of matrices")
        self._brdf = sets
        vol = (C.c_void_p * len(sets))(*[st[0].data_ptr() for st in sets])
        geo = (C.c_void_p * len(sets))(*[st[1].data_ptr() for st in sets]) if len(sets[0]) > 1 else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_plan_set_brdf(self._plan, vol, geo, len(sets), int(ldr)), "sos_plan_set_brdf")

    def set_brdf_scenarios(self, sets: np.ndarray, weights: np.ndarray, beams: np.ndarray):
        """Per-scenario Ross-Li / ocean data (sos_plan_set_brdf_scenarios): sets (S,) set index, weights (S, 2) = (f_vol, f_geo)
        or (f_glint, 0), beams (S, 2, M-1) = the beam vectors of the scenario's mode (the ocean's second is not read).
        Rewritten in place: captured graphs stay valid."""
        st = np.ascontiguousarray(sets, dtype=np.int32)
        f = np.ascontiguousarray(weights, dtype=np.float64)
        b = np.ascontiguousarray(beams, dtype=np.float64)
        if st.shape != (self.S,) or f.shape != (self.S, 2) or b.shape != (self.S, 2, self.M - 1):
            raise ValueError("set_brdf_scenarios: shapes do not match the plan")
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_plan_set_brdf_scenarios(self._plan, st.ctypes.data, f.ctypes.data, b.ctypes.data, self._stream),
                       "sos_plan_set_brdf_scenarios")

    # ------------------------------------------------------------------ ocean
    def build_glint_modes(self, wind_speed: float, n_ref: float = 1.34, n_modes: int = 1,
                          n_quad: Optional[int] = None) -> torch.Tensor:
        """Fourier modes 0 .. n_modes-1 of the Cox-Munk glint at wind speed W (m/s) and relative refractive index n_ref on
        this grid, built ON THE DEVICE (sos_build_glint_modes): a (n_modes, M, ldr) tensor, [m][c][i] =
        rho_m(mu[M+1+i], |mu[c]|) (the transposed layout the coupling reads; ldr = M-1 rounded up to even).
        ocean.glint_modes is the NumPy reference ([m][i][c])."""
        from . import brdf as BR, ocean as OC
        K, nq = int(n_modes), int(n_quad if n_quad is not None else BR.BRDF_NODES)
        M = self.M
        ldr = _align(M - 1, 2)
        R = torch.zeros((K, M, ldr), dtype=torch.float64, device=self.device)
        phi, tab = BR.node_table(nq, K)
        tab[0] = np.cos(phi)   # (the glint takes cos phi itself: it sits at phi = 0)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_build_glint_modes(self._plan, nq, phi.ctypes.data, tab.ctypes.data, K,
                                                      float(OC.slope_variance(wind_speed)), float(n_ref), R.data_ptr(), ldr,
                                                      M * ldr, self._stream), "sos_build_glint_modes")
            torch.cuda.current_stream(self.device).synchronize()   # (phi / tab are host temporaries)
        return R

    def glint_correction(self, out: torch.Tensor, geo: np.ndarray, params: np.ndarray, tau_rows: np.ndarray, beams: np.ndarray,
                         phi: np.ndarray):
        """Exact direct glint of azimuth-resolved radiance (sos_glint_correction): out (n_geo, n_rows, n_az, N) as written by
        azimuth_synthesis; per entry k: geo[k] its geometry, params[k] = (mu0, tauStar_tot, sigma^2, n_ref), tau_rows[k] tau at
        the rows, beams[k] (n_modes, M-1) the glint beam vectors of the modes summed into out."""
        ge = np.ascontiguousarray(geo, dtype=np.int32)
        par = np.ascontiguousarray(params, dtype=np.float64)
        tr = np.ascontiguousarray(tau_rows, dtype=np.float64)
        b = np.ascontiguousarray(beams, dtype=np.float64)
        ph = np.ascontiguousarray(phi, dtype=np.float64)
        n = ge.size
        n_geo, n_rows, n_az = out.shape[:3]
        if (par.shape != (n, 4) or tr.shape != (n, n_rows) or b.ndim != 3 or b.shape[0] != n or b.shape[2] != self.M - 1
                or ph.shape != (n_az,) or out.shape[3] != self.N or not out.is_contiguous()):
            raise ValueError("glint_correction: shapes do not match the plan")
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_glint_correction(self._plan, n, ge.ctypes.data, par.ctypes.data, tr.ctypes.data, n_rows,
                                                     b.ctypes.data, b.shape[1], ph.ctypes.data, n_az, n_geo, out.data_ptr(),
                                                     self._stream), "sos_glint_correction")
            torch.cuda.current_stream(self.device).synchronize()   # (the host tables are temporaries)
        return out

    def single_scatter_correction(self, out: torch.Tensor, entries: np.ndarray, P0m: np.ndarray, tables: np.ndarray,
                                  rows: Sequence[int], phi: np.ndarray):
        """Exact single scattering of azimuth-resolved radiance (sos_single_scatter_correction): out (n_geo, n_rows, n_az, N) as
        written by azimuth_synthesis at the layers `rows`; entries: _lib.SS_ENTRY_DTYPE records (plan scenario, geometry,
        phase families, rows of P0m, table offsets, g, normalisations T, weights (alb_atm, f_atm, alb_aer, f_aer)); P0m
        (n_vec, n_modes, N) the solar mode vectors the radiance was summed with; tables the tabulated phase functions
        (abscissae then values at each entry's offset); phi (n_az,)."""
        ent = np.ascontiguousarray(entries)
        p0 = np.ascontiguousarray(P0m, dtype=np.float64)
        tab = np.ascontiguousarray(tables, dtype=np.float64).reshape(-1)
        rw = np.ascontiguousarray(rows, dtype=np.int32)
        ph = np.ascontiguousarray(phi, dtype=np.float64)
        n_geo, n_rows, n_az = out.shape[:3]
        if (ent.dtype != _lib.SS_ENTRY_DTYPE or ent.ndim != 1 or p0.ndim != 3 or p0.shape[2] != self.N or rw.shape != (n_rows,)
                or ph.shape != (n_az,) or out.shape[3] != self.N or out.dtype != torch.float64 or not out.is_contiguous()):
            raise ValueError("single_scatter_correction: shapes do not match the plan")
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_single_scatter_correction(self._plan, int(ent.size), ent.ctypes.data, p0.ctypes.data, p0.shape[0],
                                                              p0.shape[1], tab.ctypes.data if tab.size else None, int(tab.size),
                                                              rw.ctypes.data, n_rows, ph.ctypes.data, n_az, n_geo, out.data_ptr(),
                                                              self._stream), "sos_single_scatter_correction")
            torch.cuda.current_stream(self.device).synchronize()   # (the host tables are temporaries)
        return out

    def azimuth_synthesis(self, I: torch.Tensor, geo: np.ndarray, weights: np.ndarray, n_geo: int, rows: Sequence[int],
                          out: torch.Tensor, accumulate: bool):
        """out[geo][r][p][:] (+)= sum over the members s of geo (ascending) of weights[s, p] * I[s, rows[r], :N]
        (sos_azimuth_synthesis).  geo (S,) int: geometry of each member, -1 = not summed; out: (n_geo, n_rows, n_az, N)."""
        ge = np.ascontiguousarray(geo, dtype=np.int32)
        w = np.ascontiguousarray(weights, dtype=np.float64)
        rw = np.ascontiguousarray(rows, dtype=np.int32)
        n_az = w.shape[1]
        if ge.shape != (self.S,) or w.shape != (self.S, n_az) or out.shape != (n_geo, rw.size, n_az, self.N) or not out.is_contiguous():
            raise ValueError("azimuth_synthesis: shapes do not match the plan")
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_azimuth_synthesis(self._plan, I.data_ptr(), ge.ctypes.data, w.ctypes.data, int(n_geo),
                                                      rw.ctypes.data, int(rw.size), int(n_az), out.data_ptr(), int(bool(accumulate)),
                                                      self._stream), "sos_azimuth_synthesis")
        return out

    # ------------------------------------------------------------------ operators
    def first_order(self, C_coef: np.ndarray, out: Optional[torch.Tensor] = None, also_into: Optional[torch.Tensor] = None) -> torch.Tensor:
        """C_coef: (S, 2, N) -- see sos_first_order in sos_b200.h.  also_into: a second field that receives the same values
        (the accumulator of the order loop: solve(..., I=also_into, I_holds_I1=True) then skips its field copy)."""
        Cc = np.ascontiguousarray(C_coef, dtype=np.float64).reshape(self.S, 2, self.N)
        out = self.new_field(zero=True) if out is None else out
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_first_order2(self._plan, Cc.ctypes.data, out.data_ptr(),
                                                 also_into.data_ptr() if also_into is not None else None, self._stream),
                       "sos_first_order")
        return out

    def first_order_from_table(self, P0tab: np.ndarray, idx: np.ndarray, weights: np.ndarray, out: Optional[torch.Tensor] = None,
                               also_into: Optional[torch.Tensor] = None) -> torch.Tensor:
        """First order with the (S, 2, N) coefficient planes assembled on the device (sos_first_order_tab): P0tab (K, N) =
        the distinct solar phase vectors of the batch, idx (S, 2) int32 = rows used by (atmosphere, aerosol), weights (S, 4) =
        (alb_atm, f_atm, alb_aer, f_aer).  Same bits as first_order() on the host-assembled planes."""
        tab = np.ascontiguousarray(P0tab, dtype=np.float64).reshape(-1, self.N)
        ix = np.ascontiguousarray(idx, dtype=np.int32).reshape(self.S, 2)
        w = np.ascontiguousarray(weights, dtype=np.float64).reshape(self.S, 4)
        out = self.new_field(zero=True) if out is None else out
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_first_order_tab(self._plan, tab.ctypes.data, int(tab.shape[0]), ix.ctypes.data, w.ctypes.data,
                                                    out.data_ptr(), also_into.data_ptr() if also_into is not None else None,
                                                    self._stream), "sos_first_order_tab")
        return out

    @staticmethod
    def table_fits(n_tab: int, S: int, N: int) -> bool:
        """sos_first_order_tab's staging constraint (include/sos_b200.h)."""
        return n_tab * N + 5 * S <= 2 * S * N

    def source(self, In1: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        out = self.new_field(zero=True) if out is None else out
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_source(self._plan, In1.data_ptr(), out.data_ptr(), self._stream), "sos_source")
        return out

    def source_rows(self, In1: torch.Tensor, out: torch.Tensor, row0: int, row1: int) -> torch.Tensor:
        """Source contraction of layers [row0, row1) only (see sos_source_rows)."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_source_rows(self._plan, In1.data_ptr(), out.data_ptr(), int(row0), int(row1), self._stream),
                       "sos_source_rows")
        return out

    def sweeps(self, J: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate_into: Optional[torch.Tensor] = None):
        out = self.new_field(zero=True) if out is None else out
        acc = accumulate_into.data_ptr() if accumulate_into is not None else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_sweeps(self._plan, J.data_ptr(), out.data_ptr(), acc, self._stream), "sos_sweeps")
        return out

    def set_columns(self, col0: int, col1: int):
        """Own only the mu columns [col0, col1) (mu-block sharding, see sos_plan_set_columns)."""
        if (int(col0), int(col1)) != (0, self.N) and self.folded:
            # column-sharded plans use the general contraction: leave fold mode (its tile plan has fold-only row classes)
            _lib.check(self.lib.sos_plan_set_folded(self._plan, None, 0, 0), "sos_plan_set_folded")
            self.folded = False
        _lib.check(self.lib.sos_plan_set_columns(self._plan, int(col0), int(col1)), "sos_plan_set_columns")
        self.col0, self.col1 = int(col0), int(col1)

    def layer_mailbox_bytes(self) -> int:
        n = C.c_size_t()
        _lib.check(self.lib.sos_layer_mailbox_bytes(self._plan, C.byref(n)), "sos_layer_mailbox_bytes")
        return int(n.value)

    def set_layers(self, rank: int, world: int, mailbox_ptrs=None, In_ptrs=None):
        """Own only a block of layers (layer-block sharding, see sos_plan_set_layers); returns its rows [row0, row1).
        mailbox_ptrs / In_ptrs: ctypes arrays of `world` device pointers (every rank's buffers as mapped here)."""
        r0, r1 = C.c_int(), C.c_int()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_plan_set_layers(self._plan, int(rank), int(world), mailbox_ptrs, In_ptrs, C.byref(r0), C.byref(r1)),
                       "sos_plan_set_layers")
        self.row0, self.row1 = int(r0.value), int(r1.value)
        return self.row0, self.row1

    def ratios(self, buf: Optional[torch.Tensor] = None, set: bool = False) -> torch.Tensor:
        """Device tensor (S, 2) of {ratio_toa, ratio_surf}; set=True writes `buf` back into the plan."""
        if buf is None:
            buf = torch.empty((self.S, 2), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_state_ratios(self._plan, buf.data_ptr(), 1 if set else 0, self._stream), "sos_state_ratios")
        return buf

    def reset(self, I1: torch.Tensor):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_reset(self._plan, I1.data_ptr(), self._stream), "sos_reset")

    def converge(self, order: int):
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_converge(self._plan, int(order), self._stream), "sos_converge")

    def results(self):
        res = (_lib.sos_result * self.S)()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_get_results(self._plan, res, self._stream), "sos_get_results")
        return res

    def solve(self, I1: torch.Tensor, max_orders: int = 10000, keep_orders: int = 0, poll_every: int = 1,
              In: Optional[torch.Tensor] = None, J: Optional[torch.Tensor] = None, I: Optional[torch.Tensor] = None,
              consume_I1: bool = False, I_holds_I1: bool = False) -> SolveResult:
        """The order loop of SOS_Aer() (SOS_Aer_main_specular.py:302-458) for the whole batch.

        I1 is not modified unless consume_I1 is set: then its buffer serves as the I_n field of the loop (one field copy
        less per solve; the caller recomputes the first order before it needs it again).  keep_orders > 0 also returns
        the first `keep_orders` fields I_n (n >= 2).  I_holds_I1: the accumulator I already holds I1 (first_order(also_into=I)).
        """
        I = self._buf("I") if I is None else I
        J = self._buf("J") if J is None else J
        orders = None
        optr = None
        if keep_orders > 0:
            orders = torch.zeros((keep_orders, self.S * self.L, self.ld), dtype=torch.float64, device=self.device)
            optr = orders.data_ptr()
        res = (_lib.sos_result * self.S)()
        In_arg = In
        for attempt in (0, 1):
            if not (I_holds_I1 and attempt == 0):
                I.copy_(I1)
            if consume_I1 and In_arg is None:
                In = I1
            else:
                In = self._buf("In") if In_arg is None else In_arg
                In.copy_(I1)
            try:
                with torch.cuda.device(self.device):
                    _lib.check(self.lib.sos_solve(self._plan, I.data_ptr(), In.data_ptr(), J.data_ptr(), optr, keep_orders,
                                                  int(max_orders), int(poll_every), res, self._stream), "sos_solve")
                break
            except _lib.SosRetry:
                # a blend reached past the columns whose raw I_n is kept; the plan now stores every row.  With
                # consume_I1 the first order is gone: the owner of I1 (BatchSolver.solve) recomputes it and calls again.
                if attempt or (consume_I1 and In_arg is None):
                    raise
        n = np.array([r.n_orders for r in res])
        return SolveResult(I, n, np.array([r.ratio_toa for r in res]), np.array([r.ratio_surf for r in res]),
                           np.array([r.status for r in res], dtype=np.uint32), orders,
                           active=np.array([r.active for r in res], dtype=np.int32))

    def quadratures(self, I: torch.Tensor, z: Optional[np.ndarray] = None, direct_scale: float = 1.0, heating: bool = True):
        """flux_up, flux_down, net_flux, diffusivity, heating_rate -- each (S, L) on the host."""
        packed = torch.zeros((5, self.S, self.L), dtype=torch.float64, device=self.device)
        outs = [packed[k] for k in range(5)]
        want_heat = heating and z is not None and self.n_regions == 3
        zc = np.ascontiguousarray(z, dtype=np.float64) if z is not None else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sos_quadratures(self._plan, I.data_ptr(), float(direct_scale),
                                                zc.ctypes.data if zc is not None else None,
                                                outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(), outs[3].data_ptr(),
                                                outs[4].data_ptr() if want_heat else None, self._stream), "sos_quadratures")
            # one D2H through a cached pinned buffer (five pageable .cpu() calls cost ~1 ms per batch)
            stage = _pinned_pair(packed.numel())[0][: packed.numel()]
            stage.copy_(packed.view(-1), non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
        host = stage.numpy().reshape(5, self.S, self.L).copy()
        return dict(flux_up=host[0], flux_down=host[1], net_flux=host[2], diffusivity=host[3],
                    heating_rate=host[4] if want_heat else None)
