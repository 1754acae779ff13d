"""Cost of the exact single scattering of azimuth-resolved radiance (solve_azimuthal(..., single_scatter='exact')) on one GPU;
one JSON line.

Workload: bench.py's 96-scenario batch on the 800 x 1002 grid (specular ground, Rayleigh atmosphere, ten mu0), with the
aerosol phase function replaced in turn by HG g = 0.85, the FWC cloud table and the EVA log-normal Mie mixture; 2 rows
(TOA, surface), 64 azimuths on [0, pi], K = 16 and 64 modes (n_quad = 2K + 1 azimuth nodes).  Per family and K (after a
warm-up of every shape):
  correction_ms   the whole correction of the mode-0 batch as solve_azimuthal runs it (azimuth._single_scatter_correction:
                  host tables, their upload and the kernel; the host-built mode vectors already cached), CUDA events
  kernel_us       single_scatter_kernel alone (torch.profiler, a run of its own)
  elements        output elements corrected (geometries x rows x azimuths x columns) and distinct series vectors uploaded
and once per family:
  synthesis_ms    sos_azimuth_synthesis of the mode-0 batch into the same output (CUDA events)
  solve_ms        the mode-0 solve, BatchSolver.solve (CUDA events)
The mode vectors m >= 1 are put into the host phase cache from one phase_modes call per (phase function, mu0) -- the same
bits as the per-mode builds of the mode members (every mode is computed independently of K) -- so that the set-up is not
timed with it.
Usage: python tools/single_scatter_time.py [--out FILE]
"""
import argparse
import dataclasses
import json
import os
import subprocess
import sys
from importlib import import_module

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
import sos_b200 as sos  # noqa: E402

AZ = import_module("sos-radiative-transfer_b200.azimuth")
DR = import_module("sos-radiative-transfer_b200.drivers")
PH = import_module("sos-radiative-transfer_b200.phase")

FAMILIES = {"hg": ("hg", 0.85), "fwc": ("fwc", 0.5), "mie": ("eva", None)}
MODES = (16, 64)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_us(fn, name, reps):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    for evt in prof.key_averages():
        if name in evt.key:
            total = getattr(evt, "device_time_total", None)
            if total is None:
                total = evt.cuda_time_total
            return dict(us=round(total / evt.count, 3), launches=int(evt.count))
    return None


def prefill(bs, K, n_quad):
    """Host mode vectors m = 1 .. K-1 of every (phase function, mu0) of the batch into drivers._PHASES."""
    seen = set()
    for sc in bs.scenarios:
        for spec in (sc.atm_phase, sc.aer_phase):
            name, g = PH.resolve(spec[0], spec[1] if len(spec) > 1 else None)
            gk = tuple(float(v) for v in g) if isinstance(g, (tuple, list)) else float(g)
            if name == "iso" or (name, gk, sc.mu0) in seen:
                continue
            seen.add((name, gk, sc.mu0))
            P0m, _ = PH.phase_modes(name, bs.M, bs.mu, K, g, mu0=sc.mu0, n_quad=n_quad, want_P=False)
            for m in range(1, K):
                DR._PHASES._P0[(name, gk, bs.M, float(sc.mu0), m, n_quad)] = P0m[m]
    return len(seen)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--scenarios", type=int, default=96)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("single_scatter_time.py needs a GPU")
    torch.cuda.set_device(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, check=True).stdout.strip()
    except Exception as e:  # (reported, not guessed)
        power = f"unavailable: {e}"
    scen = bench.make_scenarios(sos, args.scenarios)
    n_az = 64
    phi = np.linspace(0.0, np.pi, n_az)
    per = {}
    for fam, spec in FAMILIES.items():
        batch = [dataclasses.replace(sc, aer_phase=spec) for sc in scen]
        bs = sos.BatchSolver(batch)
        try:
            eng = bs.engine
            res = bs.solve()
            rws = np.array([0, bs.L - 1])
            geo = np.arange(len(batch))
            out = torch.zeros((len(batch), rws.size, n_az, eng.N), dtype=torch.float64, device=eng.device)
            rec = dict(orders_min_max=[int(res.n_orders.min()), int(res.n_orders.max())])
            rec["synthesis_ms"] = round(timed(lambda: eng.azimuth_synthesis(res.I, geo, np.ones((len(batch), n_az)), len(batch),
                                                                            rws, out, accumulate=False), args.reps), 4)
            rec["solve_ms"] = round(timed(lambda: bs.solve(), 3), 3)
            for K in MODES:
                nq = 2 * K + 1
                n_vec = prefill(bs, K, nq)

                def corr():
                    AZ._single_scatter_correction(eng, bs, geo, rws, K, nq, phi, out)
                rec[f"K{K}"] = dict(n_quad=nq, series_vectors=n_vec, elements=int(out.numel()),
                                    correction_ms=round(timed(corr, args.reps), 4),
                                    kernel_us=kernel_us(corr, "single_scatter_kernel", args.reps))
            per[fam] = rec
        finally:
            bs.engine.close()
            DR.clear_caches()
    sc0 = scen[0]
    rec = dict(tool="single_scatter_time", device=torch.cuda.get_device_name(0), power_limit=power,
               grid=[sc0.nb_layers, 2 * sc0.nb_angles], scenarios=len(scen), rows=2, azimuths=n_az,
               workload="bench.py make_scenarios, aerosol phase replaced by HG 0.85 / FWC / EVA Mie", reps=args.reps,
               families=per)
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
