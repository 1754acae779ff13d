"""Cost of the diffuse Lambert ground (surface="lambert_diffuse") on one GPU; prints one JSON line.

Workload: bench.py's 96-scenario batch on the 800 x 1002 grid (tau_aer x mu0 x omega_aer x albedo x phase sweep), with the
surface replaced by 'specular', 'lambert_readme' and 'lambert_diffuse' in turn.  Per surface (after a warm-up of every
shape):
  first_order_ms      the first order as BatchSolver.solve issues it (sos_first_order_tab: coefficient assembly, for
                      lambert_diffuse the surface pre-pass, the closed-form kernel), CUDA events over --reps calls
  kernels_us          mean device time per launch of the first-order kernels (torch.profiler, a run of its own):
                      first_order_surface_kernel is the pre-pass; first order without it = first_order_regions_kernel
  solve_ms            BatchSolver.solve (first order + order loop), CUDA events over --solve-reps calls
  scenario_orders     sum over the batch of the orders to convergence
Usage: python tools/lambert_time.py [--out FILE]
"""
import argparse
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

SURFACES = ("specular", "lambert_readme", "lambert_diffuse")
KERNELS = ("first_order_coef_kernel", "first_order_surface_kernel", "first_order_regions_kernel")


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
    """Mean device time per launch (us) of the first-order kernels over `reps` calls of fn."""
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
                out[k] = round(total / evt.count, 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--scenarios", type=int, default=96)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--solve-reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lambert_time.py needs a GPU")
    torch.cuda.set_device(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, check=True).stdout.strip()
    except Exception as e:  # (reported, not guessed)
        power = f"unavailable: {e}"
    scen = bench.make_scenarios(sos, args.scenarios)
    per = {}
    for surface in SURFACES:
        batch = [dataclasses.replace(sc, surface=surface) for sc in scen]
        bs = sos.BatchSolver(batch)
        try:
            res = bs.solve()
            acc = bs.engine.new_field(zero=True)
            fo = timed(lambda: bs.first_order(also_into=acc), args.reps)
            kus = kernel_us(lambda: bs.first_order(also_into=acc), args.reps)
            solve = timed(lambda: bs.solve(), args.solve_reps)
            per[surface] = dict(first_order_ms=round(fo, 4), kernels_us=kus, solve_ms=round(solve, 3),
                                scenario_orders=int(np.sum(res.n_orders)),
                                status_nonzero=int(np.count_nonzero(res.status)), orders_min_max=[int(res.n_orders.min()), int(res.n_orders.max())])
        finally:
            bs.engine.close()
    sc0 = scen[0]
    rec = dict(tool="lambert_time", device=torch.cuda.get_device_name(0), power_limit=power,
               grid=[sc0.nb_layers, 2 * sc0.nb_angles], scenarios=len(scen), workload="bench.py make_scenarios, surface replaced",
               reps=args.reps, solve_reps=args.solve_reps, surfaces=per)
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
