"""Timing of the azimuth-resolved solve (sos_b200.solve_azimuthal) on one GPU; prints one JSON line.

Workload: the README's EVA scenario (Rayleigh atmosphere, log-normal Mie 'eva' aerosol, specular surface) on the default
800 x 1002 grid, K = 16 Fourier modes built with n_quad = 64 azimuth nodes, radiance synthesized at 360 azimuths on the
TOA and surface rows.  Reported (CUDA events, after a warm-up of every shape):
  builder_ms          sos_build_phase_modes: all 16 modes of both phase functions (N x N matrices)
  solve_mode0_ms      the mode-0 solve (BatchSolver.solve, what solve_scenarios runs)
  solve_subbatch_ms   each sub-batch of modes 1 .. 15 (one plan each, order_cap = the mode-0 order count)
  synth_ms / synth_bytes / synth_hbm_share
                      sos_azimuth_synthesis of the largest sub-batch into the accumulated output; bytes = the member rows
                      read once + the output read and written once, over the HBM peak of the data sheet (7.7 TB/s)
Usage: python tools/azimuth_time.py [--out FILE]
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

import sos_b200 as sos  # noqa: E402
from importlib import import_module  # noqa: E402

AZ = import_module("sos-radiative-transfer_b200.azimuth")
DR = import_module("sos-radiative-transfer_b200.drivers")

HBM_PEAK = 7.7e12


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--modes", type=int, default=16)
    ap.add_argument("--n-quad", type=int, default=64)
    ap.add_argument("--n-az", type=int, default=360)
    args = ap.parse_args()
    K, nq, n_az = args.modes, args.n_quad, args.n_az
    if not torch.cuda.is_available():
        raise SystemExit("azimuth_time.py needs a GPU")
    torch.cuda.set_device(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, check=True).stdout.strip()
    except Exception as e:  # (reported, not guessed)
        power = f"unavailable: {e}"
    sc = sos.Scenario(**sos.EVA, aer_phase=("eva", None))
    rows = np.array([0, sc.nb_layers - 1])
    phi = np.linspace(0, 2 * np.pi, n_az, endpoint=False)

    # mode 0, exactly as solve_scenarios / solve_azimuthal run it
    bs0 = sos.BatchSolver([sc])
    solve0 = timed(lambda: bs0.solve(), 5)
    n0 = int(bs0.solve().n_orders[0])

    # mode builder: 16 modes of both phase functions on the plan's grid
    eng = bs0.engine
    name_aer, g_aer = sos.phase.resolve("eva")
    build = {n: timed(lambda n=n, g=g: eng.build_phase_modes(n, g, n_modes=K, n_quad=nq), 3)
             for n, g in (("rayleigh", 0.5), (name_aer, g_aer))}
    bs0.engine.close()

    # modes 1 .. K-1: the sub-batches solve_azimuthal forms
    members = [dataclasses.replace(sc, atm_phase=AZ._mode_spec(sc.atm_phase, m, nq), aer_phase=AZ._mode_spec(sc.aer_phase, m, nq))
               for m in range(1, K) if not (AZ._vanishes(sc.atm_phase, m) and AZ._vanishes(sc.aer_phase, m))]
    subs = DR.split_for_plan_limits(members, range(len(members)), max_phases=AZ.MODE_PHASES_PER_PLAN)
    sub_ms, synth = [], None
    for sub in subs:
        bs = sos.BatchSolver([members[j] for j in sub], order_caps=[n0] * len(sub))
        res = bs.solve(max_orders=n0)
        assert np.all(res.n_orders == n0) and np.all(res.status == 0)
        sub_ms.append(timed(lambda: bs.solve(max_orders=n0), 3))
        if synth is None or len(sub) > synth[0]:
            e = bs.engine
            out = torch.zeros((1, rows.size, n_az, e.N), dtype=torch.float64, device=e.device)
            w = np.stack([2 * np.cos((1 + j) * phi) for j in sub])
            ms = timed(lambda: e.azimuth_synthesis(res.I, np.zeros(len(sub), dtype=np.int32), w, 1, rows, out, True), 50)
            nbytes = 8 * e.N * rows.size * (len(sub) + 2 * n_az)
            synth = (len(sub), ms, nbytes)
        bs.engine.close()
    rec = dict(tool="azimuth_time", device=torch.cuda.get_device_name(0), power_limit=power, grid=[sc.nb_layers, 2 * sc.nb_angles],
               scenario="EVA (rayleigh + eva Mie, specular)", n_modes=K, n_quad=nq, n_az=n_az, mode0_orders=n0,
               builder_ms={k: round(v, 3) for k, v in build.items()}, solve_mode0_ms=round(solve0, 3),
               solve_subbatch_ms=[round(v, 3) for v in sub_ms], subbatch_modes=[len(s) for s in subs],
               synth_members=synth[0], synth_ms=round(synth[1], 4), synth_bytes=synth[2],
               synth_hbm_share=round(synth[2] / (synth[1] * 1e-3) / HBM_PEAK, 4))
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
