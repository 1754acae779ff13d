"""Cost of the ocean ground (surface="ocean") against the diffuse Lambert and Ross-Li grounds on one GPU; one JSON line.

Workload: bench.py's 96-scenario batch on the 800 x 1002 grid with grd_alb = 0.02 and the surface replaced by
'lambert_diffuse', by 'rossli' (f_vol = 0.1, f_geo = 0.03) and by 'ocean' (four wind speeds, 1 / 3 / 7 / 12 m/s, in turn
over the batch: four glint matrix sets).  Per surface (after a warm-up of every shape):
  builder_ms          ocean: SosEngine.build_glint_modes for 1 and for 64 modes (CUDA events, one call each after a warm-up)
  correction_ms       ocean: sos_glint_correction of 64 modes for the 96 geometries, 2 rows and 64 azimuths (CUDA events)
  kernels_us          mean device time per launch (torch.profiler, a run of its own over --solve-reps solves) of the surface
                      pre-pass first_order_surface_kernel, the closed-form first order and the carry kernel of the sweeps
                      (sweep_carry_kernel: where the BRDF / glint mat-vecs run, once per active scenario and order)
  sweeps_ms_per_order the layer sweeps of one order (sos_set_profiling class 1: every sweep launch of the order) averaged
                      over the orders of a solve -- profiling runs the order loop without CUDA graphs
  solve_ms            BatchSolver.solve (first order + order loop, graphs on), CUDA events over --solve-reps calls
  scenario_orders     sum over the batch of the orders to convergence
Usage: python tools/ocean_time.py [--out FILE]
"""
import argparse
import ctypes as C
import dataclasses
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
import sos_b200 as sos  # noqa: E402

SURFACES = {"lambert_diffuse": {}, "rossli": dict(brdf_vol=0.1, brdf_geo=0.03), "ocean": {}}
WINDS = (1.0, 3.0, 7.0, 12.0)
KERNELS = ("first_order_surface_kernel", "first_order_regions_kernel", "sweep_carry_kernel")


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


def kernel_us(fn, reps):
    """Mean device time per launch (us) and launch count of the named kernels over `reps` calls of fn."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for evt in prof.key_averages():
        for k in KERNELS:
            if k in evt.key:
                total = getattr(evt, "device_time_total", None)
                if total is None:
                    total = evt.cuda_time_total
                out[k] = dict(us=round(total / evt.count, 3), launches=int(evt.count))
    return out


def sweeps_per_order(bs):
    """ms per order of the sweeps (profiling class 1), averaged over one solve."""
    eng = bs.engine
    lib = eng.lib
    sos._lib.check(lib.sos_set_profiling(eng._plan, 1), "sos_set_profiling")
    try:
        bs.solve()
        ms = (C.c_double * 4)()
        spans = (C.c_longlong * 4)()
        sos._lib.check(lib.sos_get_profile(eng._plan, ms, spans, eng._stream), "sos_get_profile")
    finally:
        sos._lib.check(lib.sos_set_profiling(eng._plan, 0), "sos_set_profiling")
    return round(ms[1] / max(1, spans[1]), 4), int(spans[1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--scenarios", type=int, default=96)
    ap.add_argument("--solve-reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ocean_time.py needs a GPU")
    torch.cuda.set_device(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, check=True).stdout.strip()
    except Exception as e:  # (reported, not guessed)
        power = f"unavailable: {e}"
    scen = bench.make_scenarios(sos, args.scenarios)
    per = {}
    for surface, weights in SURFACES.items():
        batch = [dataclasses.replace(sc, surface=surface, grd_alb=0.02, **weights) for sc in scen]
        if surface == "ocean":
            batch = [dataclasses.replace(sc, wind_speed=WINDS[i % len(WINDS)]) for i, sc in enumerate(batch)]
        bs = sos.BatchSolver(batch)
        try:
            res = bs.solve()
            rec = {}
            if surface == "ocean":
                eng = bs.engine
                rec["builder_ms"] = {str(k): round(timed(lambda k=k: eng.build_glint_modes(5.0, n_modes=k), 1), 3) for k in (1, 64)}
                K, rows, phi = 64, np.array([0, bs.L - 1]), np.linspace(0.0, np.pi, 64)
                out = torch.zeros((len(batch), rows.size, phi.size, eng.N), dtype=torch.float64, device=eng.device)
                par = np.array([[sc.mu0, sc.tauStar_atm + sc.tauStar_aer, float(sos.ocean.slope_variance(sc.wind_speed)),
                                 sc.ocean_index] for sc in batch])
                beams = np.stack([sos.drivers.glint_beam(bs.M, bs.mu, sc, K) for sc in batch])
                geo = np.arange(len(batch))
                rec["correction_ms"] = round(timed(lambda: eng.glint_correction(out, geo, par, bs.tau[:, rows], beams, phi), 3), 3)
            rec["kernels_us"] = kernel_us(lambda: bs.solve(), args.solve_reps)
            rec["sweeps_ms_per_order"], rec["sweep_spans"] = sweeps_per_order(bs)
            rec["solve_ms"] = round(timed(lambda: bs.solve(), args.solve_reps), 3)
            rec.update(scenario_orders=int(np.sum(res.n_orders)), status_nonzero=int(np.count_nonzero(res.status)),
                       orders_min_max=[int(res.n_orders.min()), int(res.n_orders.max())])
            per[surface] = rec
        finally:
            bs.engine.close()
    sc0 = scen[0]
    rec = dict(tool="ocean_time", device=torch.cuda.get_device_name(0), power_limit=power,
               grid=[sc0.nb_layers, 2 * sc0.nb_angles], scenarios=len(scen),
               workload="bench.py make_scenarios, grd_alb 0.02, surface replaced (rossli: f_vol 0.1, f_geo 0.03; "
                        "ocean: wind speeds 1 / 3 / 7 / 12 m/s in turn, n = 1.34)",
               solve_reps=args.solve_reps, surfaces=per)
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
