#!/usr/bin/env python
"""bench.py -- scattering-order updates/s of the SOS_AER hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--scenarios S] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[4], the critical-albedo style batch sweep): S independent
three-region scenarios per GPU on the reference's default grid (800 layers x 1002 mu), spanning
tau_aer x mu0 x omega_aer x surface albedo x aerosol phase function (HG / log-normal Mie stand-in / FWC); every GPU solves its own S
scenarios with no data-path collective (scaling: weak).  With N GPUs the job is members 0 .. N*S-1 of the sweep, dealt so that
every rank gets a batch of the same make-up (job_deal: sorted by cost, serpentine rounds; first by a cost proxy, then by the
orders to convergence a pilot solve measured -- the line's details.dealing says so).  A "step" is one whole solve of the batch:
closed-form first order + the order loop to In/I < 1e-4 for every scenario.

  metric  = sum over scenarios and orders n >= 2 of L*N^2  /  time     (SURVEY.md 8d)
  value   : inputs already resident in HBM (plan, phase operands, coefficients uploaded before)
  e2e     : the public API call with HOST scenario values in / NumPy out per step on a resident plan: BatchSolver.update
            (tau profiles, per-scenario records, the table of solar phase vectors the device assembles the first-order
            coefficients from: H2D), solve, D2H of the flux / diffusivity / heating-rate profiles, order counts and TOA
            net flux of every scenario (what a forcing sweep returns; the reference's SOS_Aer_radiative_forcing returns one
            float per solve).  new_plan_per_batch_ms / cold_ms: the same with a new plan per batch / from a cold process
  roofline: the dominant kernel of the timed steps, timed with CUDA events on the launching stream inside them.  With a
            Rayleigh atmosphere (the default workload) that is the apply pass of the layer sweeps (sweep_apply2_kernel: HBM
            bound, peak = MEASURED_PEAKS.json hbm_gbs): the molecular rows rebuild their source from two coefficients per
            row, so its algorithmic traffic is the read-modify-write of I (16 B per element) there and J + I_n + I (32 B)
            on the aerosol rows.  The whole sweep class (local + carry + apply + zone) and the dense contraction of the
            aerosol rows (jn_gemm_fold_kernel, FP64 DMMA, against the DMMA throughput measured in the same run) are
            reported next to it.
  cpu_baseline / --impl reference: the NumPy oracle port of the reference algorithm
            (oracle/sos_oracle.py, method="slices") on the host cores, bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L_DEFAULT, M_DEFAULT = 800, 501
WORKLOAD = "critical-albedo batch sweep (BASELINE configs[4]): S specular scenarios/GPU, 800x1002 grid"


PHASES_NOTE = "HG(0.5) / log-normal Mie mixture (EVA aerosol, host Lorenz-Mie stand-in: miepython absent) / FWC table"


def workload_config(S):
    """`config` of the JSON line: identical in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "scenarios_per_gpu": S, "layers": L_DEFAULT, "mu_columns": 2 * M_DEFAULT,
            "phase_functions": PHASES_NOTE, "convergence": "In/I < 1e-4 at TOA and surface (every scenario to its own order)"}


def cost_proxy(sc):
    """Orders to convergence grow with the aerosol optical depth x single-scattering albedo and with the ground albedo."""
    return sc.tauStar_aer * sc.alb_aer + 0.2 * sc.grd_alb


def job_deal(sos, S, world, L=L_DEFAULT, M=M_DEFAULT, cost=None):
    """The world*S members (0 .. world*S - 1) of the sweep a multi-GPU job solves, and who solves which: members sorted by
    cost (the proxy, or `cost[i]` = measured orders to convergence with the proxy as the tie-break) and dealt in serpentine
    rounds -- 0 .. world-1, then world-1 .. 0, so that no rank always gets the costliest member of a round.  Every rank gets
    a batch of the same make-up: the step time of the job is the slowest rank's.  Returns (job, [members of rank r])."""
    job = make_scenarios(sos, world * S, 0, L, M)
    if cost is None:
        key = lambda i: (-cost_proxy(job[i]), i)
    else:
        key = lambda i: (-cost[i], -cost_proxy(job[i]), i)
    order = sorted(range(world * S), key=key)
    return job, [[order[r * world + (rank if r % 2 == 0 else world - 1 - rank)] for r in range(S)] for rank in range(world)]


def redeal_by_orders(sos, S, world, rank, n_orders, overrun, dist, torch, dev, L=L_DEFAULT, M=M_DEFAULT):
    """Second deal of a multi-GPU job, by measured cost: `n_orders` / `overrun` are this rank's per-scenario orders to
    convergence and blend-overrun bits from a pilot solve of the FIRST deal (job_deal by the proxy).  One all-gather of
    2*S integers per rank tells every rank every member's count; all ranks then compute the same second deal.  Returns
    (this rank's scenarios, their overrun bits)."""
    job, deals = job_deal(sos, S, world, L, M)
    loc = torch.tensor(np.stack([np.asarray(n_orders, dtype=np.int64), np.asarray(overrun, dtype=np.int64)]), device=dev)
    got = [torch.empty_like(loc) for _ in range(world)]
    dist.all_gather(got, loc)
    n_of, ov = np.zeros(world * S, dtype=np.int64), np.zeros(world * S, dtype=np.int64)
    for r in range(world):
        g = got[r].cpu().numpy()
        n_of[deals[r]], ov[deals[r]] = g[0], g[1]
    _, deals = job_deal(sos, S, world, L, M, cost=n_of)
    return [job[i] for i in deals[rank]], ov[deals[rank]]


def make_scenarios(sos, S, rank=0, L=L_DEFAULT, M=M_DEFAULT, world=1):
    """Deterministic sweep tau_aer x mu0 x omega_aer x albedo x phase (SURVEY.md 8d config 5).

    world == 1: members rank*S .. rank*S + S - 1 of the sweep.  world > 1 (bench.py --gpus N): rank's share of the job's
    world*S members, see job_deal -- how the full sweep is dealt, too."""
    if world > 1:
        job, deals = job_deal(sos, S, world, L, M)
        return [job[i] for i in deals[rank]]
    taus = np.linspace(0.0075, 0.5, 10)
    mu0s = np.linspace(0.1, 1.0, 10)
    oms = np.linspace(0.7, 1.0, 10)
    albs = (0.05, 0.15, 0.3)
    # phase-function axis of BASELINE configs[4]: HG / Mie / FWC (Mie = the EVA log-normal mixture from the host stand-in)
    phases = (("hg", 0.5), ("mie_lognormal", sos.EVA_AEROSOL), ("fwc", 0.0))
    out = []
    for i in range(S):
        k = rank * S + i
        out.append(sos.Scenario(
            nb_layers=L, nb_angles=M, tauStar_atm=0.124,
            tauStar_aer=float(taus[k % 10]), mu0=float(mu0s[(k // 10 + 3 * k) % 10]),
            alb_aer=float(oms[(k // 100 + 7 * k) % 10]), grd_alb=float(albs[(k // 3 + k) % 3]),
            atm_phase=("rayleigh", 0.0), aer_phase=phases[k % 3], surface="specular"))
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.

    nvidia-smi takes a few hundred ms to start, so the sampler is started before the warm-up and
    every line is stamped on arrival; stop(t0, t1) keeps the samples that fall inside [t0, t1]."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)  # let the last in-window sample arrive
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, r in self.rows:
            if ts < t0 or ts > t1 + 0.1:
                continue
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


_CPU_CACHE = {}


def cpu_port_inputs(L, M, seed_rank):
    """Inputs of one workload scenario for the NumPy port (built once per process, untimed)."""
    key = (L, M, seed_rank)
    if key not in _CPU_CACHE:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import sos_oracle as so
        import sos_b200 as sos
        scen = make_scenarios(sos, 1, seed_rank, L, M)[0]
        mu = so.mu_grid(M)
        P0a, Pa = sos.phase_matrices("rayleigh", M, mu, scen.mu0)
        P0e, Pe = sos.phase_matrices(scen.aer_phase[0], M, mu, scen.mu0, scen.aer_phase[1])
        sc = so.Scenario(mu0=scen.mu0, nb_layers=L, nb_angles=M, tauStar_atm=scen.tauStar_atm,
                         tauStar_aer=scen.tauStar_aer, grd_alb=scen.grd_alb, alb_aer=scen.alb_aer, surface="specular")
        tau, z, iu, idn = sc.geometry()
        I1 = so.first_order_regions(sc, tau, mu, iu, idn, P0a, P0e)
        lay = so.driver_layout(sc, tau, mu, iu, idn)
        _CPU_CACHE[key] = (so, sc, mu, iu, idn, Pa, Pe, lay, I1)
    return _CPU_CACHE[key]


def cpu_port_sample(orders=2, L=L_DEFAULT, M=M_DEFAULT, seed_rank=0):
    """One scenario of the workload through the NumPy port ("slices" = the reference's O(L^2 N)
    scheme): phase matrices and first order untimed, `orders` scattering orders timed.
    orders == 0 only builds the inputs.  Returns (units, seconds)."""
    so, sc, mu, iu, idn, Pa, Pe, lay, I1 = cpu_port_inputs(L, M, seed_rank)
    In = I1
    t0 = time.perf_counter()
    for _ in range(orders):
        J = so.source_regions(sc, In, mu, iu, idn, Pa, Pe)
        In = so.order_sweeps(lay, J, method="slices")
    dt = time.perf_counter() - t0
    return orders * L * (2 * M) ** 2, dt


def _cpu_worker(args):
    # every pool worker keeps ONE scenario of the workload (chosen by its worker index), so the inputs
    # built in the untimed first round are the ones the timed rounds reuse
    import multiprocessing as mp
    ident = mp.current_process()._identity
    orders, L, M, _ = args
    return cpu_port_sample(orders, L, M, ident[0] - 1 if ident else 0)


def run_reference(args):
    """--impl reference: the reference algorithm's CPU port on all host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 32))
    orders = 1
    L = args.cpu_layers
    with mp.get_context("spawn").Pool(procs) as pool:
        # untimed: imports, phase matrices and first order of every worker's scenario (chunksize 1 and as
        # many tasks as workers: each worker builds, and later reuses, its own scenario)
        pool.map(_cpu_worker, [(0, L, M_DEFAULT, i) for i in range(procs)], chunksize=1)
        times = []
        units = 0
        for _ in range(args.steps):
            t0 = time.perf_counter()
            res = pool.map(_cpu_worker, [(orders, L, M_DEFAULT, i) for i in range(procs)], chunksize=1)
            times.append(time.perf_counter() - t0)
            units = sum(r[0] for r in res)
    ms = 1e3 * float(np.mean(times))
    val = units / (ms * 1e-3)
    sample = (f"{procs} processes x 1 scenario x {orders} order(s) of the NumPy port (method='slices') on a "
              f"{L}x{2 * M_DEFAULT} grid per step; the port vectorises over mu what the reference loops over in Python")
    emit(({
        "impl": "reference", "metric": "scattering-order updates/s", "value": val, "unit": "updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.scenarios),
        "details": {"grid": [L, 2 * M_DEFAULT], "note": "CPU sample uses the workload's scenarios; cost per order is O(L^2 N) in "
                    "the reference scheme, so a reduced L flatters the CPU"},
        "cpu_baseline": {"value": val, "unit": "updates/s", "cores": procs, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def thick_record(args, sos, torch, dist, dev, rank, world, W, steps):
    """BASELINE configs[3]: optically thick FWC cloud layer (tau* = 30, omega = 0.9) on ONE large grid
    (10 000 layers x 1024 mu), run to In/I < 1e-4; for N > 1 the grid is sharded by layer blocks (the ranks exchange scan
    aggregates, halo rows and ratios by stores into each other's memory from inside the graphed order loop; --thick-sharding
    mu: by mu blocks, the contraction reading the peers' I_n blocks by TMA over NVLink) -- strong scaling, with the one-GPU
    time of the same solve measured in the same run.  Returns the record (rank 0) or None."""
    L, M, tau_star, mu0, alb = 10000, 512, 30.0, 0.5, 0.9
    N = 2 * M
    mu = sos.mu_grid(M)
    tau = np.linspace(0, tau_star, L)
    w = sos.extrapolation_width(tau_star, M)
    coef = [sos.ScenarioCoefficients(mu0=mu0, grd_alb=0.0, tauStar_tot=tau_star, coef_atm=alb, extrap_width=(w, w, w))]
    # N > 1: layer blocks (the default) or mu blocks; the sharded plan and its one-GPU reference use the same scan chunks
    chunk_rows = args.thick_chunk_rows if world > 1 else 0
    eng = sos.SosEngine(mu, tau[None], coef, [0, L], sos._lib.SURFACE_NONE, device=dev, chunk_rows=chunk_rows)
    phase = "fwc"
    P, _ = eng.build_phase_matrix(phase)                      # built on the device
    eng.set_phase([P])
    Cc = np.zeros((1, 2, N))
    Cc[0, 0] = alb * sos.phase_P0(phase, M, mu, mu0)
    I1 = eng.first_order(Cc)
    layered = world > 1 and args.thick_sharding == "layers"
    solver = peers = None
    if layered:
        solver = sos.LayerShardedSolver(eng, rank, world)
    elif world > 1:
        blocks = sos.mu_blocks(N, M, world, M - w - 5)
        solver = sos.MuShardedSolver(eng, blocks, rank)
        peers = sos.PeerFields(eng, rank, world)

    def step():
        if world == 1:
            r = eng.solve(I1, max_orders=args.thick_orders, poll_every=8)
            return int(r.n_orders[0]), int(r.status[0])
        if layered:
            I, res = solver.solve(I1, max_orders=args.thick_orders)   # (incl. the final gather of the row blocks of I)
        else:
            I, res = solver.solve_p2p(I1, peers, max_orders=args.thick_orders)
        return int(res[0].n_orders), int(res[0].status)

    for _ in range(W):
        n, status = step()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(dev.index)
    sampler.start()
    time.sleep(0.4)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * steps)]
    t0 = time.perf_counter()
    for k in range(steps):
        ev[2 * k].record()
        n, status = step()
        ev[2 * k + 1].record()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t1 = time.perf_counter()
    clocks = sampler.stop(t0, t1)
    ms = float(np.mean([ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(steps)]))
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # the same solve unsharded on one GPU (rank 0), for the speed-up and the parity statement: a fresh engine with the folded
    # contraction; the layer-sharded plan uses the same scan chunks, so its result must equal this one bit for bit
    ms1 = None
    bit_identical = None
    if world > 1:
        if rank == 0:
            ref = sos.SosEngine(mu, tau[None], coef, [0, L], sos._lib.SURFACE_NONE, device=dev, chunk_rows=chunk_rows)
            ref.set_phase([P])
            J1 = ref.first_order(Cc)
            r1 = ref.solve(J1, max_orders=args.thick_orders, poll_every=8)
            if layered:
                bit_identical = bool(torch.equal(r1.I.view(-1, ref.ld)[:L, :N], solver._I.view(-1, eng.ld)[:L, :N]))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record()
            ref.solve(J1, max_orders=args.thick_orders, poll_every=8)   # (as in the sharded step: the first order is computed outside)
            e1.record()
            torch.cuda.synchronize(dev)
            ms1 = float(e0.elapsed_time(e1))
            ref.close()
        dist.barrier()
    units = (n - 1) * L * N * N
    if peers is not None:
        torch.cuda.synchronize(dev)
        dist.barrier()
        peers.close()
    eng_folded = bool(eng.folded)
    if layered:
        solver.close()
    eng.close()
    if rank != 0:
        return None
    rec = {
        "metric": "scattering-order updates/s", "value": units / (ms * 1e-3), "unit": "updates/s", "n_gpus": world,
        "steps": steps, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "thick FWC cloud layer (BASELINE configs[3]): one 10000x1024 grid, tau*=30, omega=0.9, "
                               "to In/I<1e-4", "orders": n, "status": status, "ms_per_order": ms / max(n - 1, 1),
                   "sharding": "none" if world == 1 else (
                       "layer blocks of %d rows; chunk aggregates, halo rows and ratios exchanged by peer-memory stores + flags inside the "
                       "graphed order loop (no NCCL on the data path)" % (L // world) if layered else
                       "mu blocks of %d columns, contraction reads peer blocks by TMA over NVLink" % (N // world)),
                   "contraction": "folded" if (eng_folded and (world == 1 or layered)) else "general",
                   "l2": "working set 4 x 82 MB fields + operand > 126 MB L2"},
        "clocks": clocks}
    if ms1 is not None:
        rec["one_gpu_ms"] = ms1
        rec["speedup_vs_1gpu"] = ms1 / ms
    if bit_identical is not None:
        rec["bit_identical_to_unsharded"] = bit_identical
    return rec


def run_thick(args, sos, torch, dist, dev, rank, world, W):
    rec = thick_record(args, sos, torch, dist, dev, rank, world, W, args.steps)
    if rank == 0:
        emit(rec)


_REAL_STDOUT = None


def emit(obj):
    """The one JSON line, on the process's real stdout (see main: libraries may chat on fd 1)."""
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


DUMP_SAMPLE = 1 << 20   # elements of the radiance field --dump-outputs writes: 2 x 8 MB (values and their indices)


def dump_outputs(dirname, res, S, L, N, torch):
    """--dump-outputs: what a caller of BatchSolver.solve received from the last timed step, as float64 DIR/<name>.npy, so
    that two builds can be compared output for output.  The (S, L, N) radiance field (615 MB at the default size) is
    written as a fixed sample: I_sample at the flat (S, L, N) indices I_sample_index, drawn by a seeded generator.  The
    per-scenario arrays (orders to convergence, last TOA / surface convergence ratios, status bits, still-active flags) are
    written whole."""
    os.makedirs(dirname, exist_ok=True)
    flat = np.sort(np.random.default_rng(0).choice(S * L * N, size=min(DUMP_SAMPLE, S * L * N), replace=False))
    ld = res.I.shape[-1]                                     # the device field pads every row of N values to ld
    padded = torch.from_numpy((flat // N) * ld + flat % N).to(res.I.device)
    out = {"I_sample": res.I.reshape(-1)[padded].cpu().numpy(), "I_sample_index": flat}
    for name in ("n_orders", "ratio_toa", "ratio_surf", "status", "active"):
        out[name] = getattr(res, name)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    # stdout carries exactly one JSON line: anything a library prints on fd 1 (NCCL prints its version there when
    # NCCL_DEBUG is set) goes to stderr instead
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scenarios", type=int, default=96, help="scenarios per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-layers", type=int, default=800)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--workload", default="sweep", choices=["sweep", "thick"],
                    help="sweep (default): BASELINE configs[4] batch; thick: configs[3], one 10000x1024 grid, mu-sharded for N>1")
    ap.add_argument("--thick-orders", type=int, default=300, help="order cap of the thick workload")
    ap.add_argument("--thick-sharding", default="layers", choices=["layers", "mu"], help="N > 1: how the one large grid is split over the GPUs")
    ap.add_argument("--thick-chunk-rows", type=int, default=0, help="N > 1, layer blocks: rows per scan chunk of the sharded plan (0: the library's choice, as on one GPU)")
    ap.add_argument("--no-secondary", dest="secondary", action="store_false", help="N > 1: skip the mu-sharded thick-cloud record")
    ap.add_argument("--full-sweep", type=int, default=9984, help="solves of the full configs[4] sweep reported as full_sweep (0: skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="sweep workload: write what the last timed step returned as "
                    "DIR/<name>.npy (rank 0; a fixed sample of the radiance field, see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "sweep"):
        ap.error("--dump-outputs covers the sweep workload of --impl ours")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    import sos_b200 as sos

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(3, args.warmup)
    if args.workload == "thick":
        run_thick(args, sos, torch, dist, dev, rank, world, W)
        if world > 1:
            dist.destroy_process_group()
        return
    S, L, M = args.scenarios, L_DEFAULT, M_DEFAULT
    N = 2 * M

    scen = make_scenarios(sos, S, rank, world=world)
    bs = sos.BatchSolver(scen, device=dev)       # plan + phase operands resident
    # scenarios on which the reference itself would die with IndexError (blend-search overrun, Q11)
    # are not valid workload members: swap their aerosol phase function for HG(0.7) once, up front
    res0 = bs.solve(poll_every=2)
    st = res0.status
    dealt_by = "the cost proxy tau_aer*omega_aer + 0.2*albedo"
    if world > 1:
        # second deal, by measured cost: the orders to convergence of this pilot solve (every rank learns every member's)
        scen, st = redeal_by_orders(sos, S, world, rank, res0.n_orders, st & 1, dist, torch, dev)
        bs.engine.close()
        bs = sos.BatchSolver(scen, device=dev)
        dealt_by = "their orders to convergence (measured by a pilot solve of the first deal, which went by the cost proxy tau_aer*omega_aer + 0.2*albedo)"
    n_swapped = int(np.sum((st & 1) != 0))
    if n_swapped:
        import dataclasses
        scen = [dataclasses.replace(sc, aer_phase=("hg", 0.7)) if (st[i] & 1) else sc for i, sc in enumerate(scen)]
        bs.engine.close()
        bs = sos.BatchSolver(scen, device=dev)
    eng = bs.engine
    lib = sos._lib.load()
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)  # 256 MB > 126 MB L2

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step_resident():
        res = bs.solve(poll_every=2)
        return res

    # ---------------- device-resident timing ----------------
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(W):
        res = step_resident()
    units_per_step = int(np.sum(res.n_orders - 1)) * L * N * N
    n_orders = res.n_orders.copy()
    barrier()
    l0 = eng.launches
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps)]
    barrier()
    t_begin = time.perf_counter()
    t_wall = t_begin
    for k in range(args.steps):
        flush.zero_()                                  # L2 flush between timed iterations (untimed)
        ev[2 * k].record()
        res = step_resident()
        ev[2 * k + 1].record()
    barrier()
    t_end = time.perf_counter()
    t_wall = t_end - t_wall
    clocks = sampler.stop(t_begin, t_end)
    launches = eng.launches - l0
    if args.dump_outputs and rank == 0:               # before the next solve overwrites the field
        dump_outputs(args.dump_outputs, res, S, L, N, torch)
    # per-kernel times: the SAME K steps once more with CUDA-event spans around every kernel class (on the launching
    # stream).  The spans cost a few percent and switch the order loop from graph replays to single launches, so the
    # headline pass above runs without them; step_ms_spans reports what this pass took.
    import ctypes as C
    lib.sos_set_profiling(eng._plan, 1)
    ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps)]
    for k in range(args.steps):
        flush.zero_()
        ev2[2 * k].record()
        step_resident()
        ev2[2 * k + 1].record()
    barrier()
    ms4 = (C.c_double * 4)()
    sp4 = (C.c_longlong * 4)()
    lib.sos_get_profile(eng._plan, ms4, sp4, None)
    lib.sos_set_profiling(eng._plan, 0)
    step_ms_spans = float(np.mean([ev2[2 * k].elapsed_time(ev2[2 * k + 1]) for k in range(args.steps)]))
    step_ms = float(np.mean([ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(args.steps)]))
    t = torch.tensor([step_ms], dtype=torch.float64, device=dev)
    u = torch.tensor([float(units_per_step)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(u, op=dist.ReduceOp.SUM)
    step_ms_max, units_all = float(t.item()), float(u.item())
    value = units_all / (step_ms_max * 1e-3)
    # every rank's own step time and work (the ranks solve DIFFERENT batches of the sweep: the slowest one sets the time)
    per_rank = None
    if world > 1:
        mine = torch.tensor([step_ms, float(units_per_step) / (L * (2 * M) ** 2)], dtype=torch.float64, device=dev)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {"ms_per_step": [round(float(x[0]), 4) for x in allr], "scenario_orders_per_step": [int(round(float(x[1]))) for x in allr]}

    # ---------------- roofline of the dominant kernel ----------------
    ms = [float(x) for x in ms4]
    spans = [int(x) for x in sp4]
    gemm_ms, gemm_launches = ms[0], spans[0]          # source contraction (all its launches of an order)
    sweep_ms, sweep_spans = ms[1], spans[1]           # the four sweep kernels of an order
    apply_ms, apply_launches = ms[2], spans[2]        # ... the apply pass alone
    dense_ms, dense_launches = ms[3], spans[3]        # the dense DMMA kernel of the contraction alone
    so_total = float(np.sum(n_orders - 1)) * args.steps            # scenario-orders inside the timed steps
    folded = bool(eng.folded)
    generated = bool(eng.generated_source)
    n_aer = int(bs.idx_down + 1 - bs.idx_up) if generated else L   # rows whose J is materialised (aerosol layer)
    hbm_peak, hbm_src = 6650.0, "fallback of /opt/skills/guides/B200_PROFILING.md (MEASURED_PEAKS.json absent)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            hbm_peak, hbm_src = float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except (OSError, KeyError, ValueError):
        pass
    pk = C.c_double()
    lib.sos_fp64_peak(1, 3, C.byref(pk))
    pk_dfma = C.c_double()
    lib.sos_fp64_peak(0, 3, C.byref(pk_dfma))
    fp64_peak = max(pk.value, pk_dfma.value)

    def ncu_traffic(fname, launches):
        """DRAM bytes per launch from the committed `ncu --set full` capture (all 96 scenarios active), scaled to the
        average number of active scenarios per timed launch."""
        try:
            with open(os.path.join(ROOT, "profiles", fname)) as f:
                tj = json.load(f)
            active = so_total / max(launches, 1)
            return (tj["dram_bytes_per_active_scenario"] * active,
                    "dram__bytes_read+write per launch from profiles/%s (%.3e B at %d active scenarios; algorithmic %.3e B) "
                    "scaled to %.1f active scenarios per timed launch" % (fname, tj["dram_bytes_per_launch"], tj["scenarios"],
                                                                          tj["algorithmic_bytes_per_launch"], active))
        except (OSError, KeyError, ValueError):
            return None, None

    # apply pass: 16 B per element where the source is rebuilt (read + write of I), 32 B where J is read and I_n kept
    apply_bytes = so_total * N * (16.0 * (L - n_aer) + 32.0 * n_aer)
    sweep_class_bytes = apply_bytes + (so_total * N * 8.0 * n_aer)        # + the local pass's read of J on the dense rows
    # dense contraction: FLOPs of the kernel that ran (folded: N^2 per row, general: 2 N^2), rows it ran on
    dense_rows = n_aer if (generated or any(int(r) for r in getattr(eng, "lowrank", []))) else L
    dense_flops = so_total * dense_rows * float(N) * N * (1.0 if folded else 2.0)
    d_ms = dense_ms if dense_launches else gemm_ms
    atr, anote = ncu_traffic("r02_ncu_apply_traffic.json", apply_launches)
    dtr, dnote = ncu_traffic("r02_ncu_dense_traffic.json", dense_launches or gemm_launches)
    contraction = {
        "bound": "tensor",
        "kernel": "jn_gemm_fold_kernel (FP64 DMMA m8n8k4; %d aerosol rows per scenario, premixed folded operands)" % dense_rows if folded
                  else "jn_gemm_dmma_kernel (FP64 DMMA m8n8k4)",
        "achieved": dense_flops / (d_ms * 1e-3) * 1e-12 if d_ms > 0 else None, "peak": fp64_peak, "unit": "TFLOP/s",
        "frac": (dense_flops / (d_ms * 1e-3) * 1e-12 / fp64_peak) if (d_ms > 0 and fp64_peak) else None,
        "traffic": dtr, "traffic_source": dnote,
        "flops_model": "%s FLOP per dense row (folded: two M x M contractions per row); rows outside the aerosol layer need no "
                       "contraction kernel (their source is rebuilt from two projections per row inside the sweeps)" % ("N^2" if folded else "2 N^2"),
        "peak_source": "FP64 DMMA m8n8k4 loop measured on this GPU in this run (sos_fp64_peak); MEASURED_PEAKS.json has no FP64 "
                       "entry; DFMA loop measured %.1f TFLOP/s" % pk_dfma.value,
        "ms_per_launch": d_ms / max(dense_launches or gemm_launches, 1), "launches": dense_launches or gemm_launches,
        "share_of_step": gemm_ms / (step_ms_spans * args.steps),
    }
    sweeps_class = {
        "kernels": "sweep_local + sweep_carry + sweep_apply2 + sweep_zone", "ms_per_order": sweep_ms / max(sweep_spans, 1),
        "achieved": sweep_class_bytes / (sweep_ms * 1e-3) * 1e-9 if sweep_ms > 0 else None, "unit": "GB/s",
        "frac": (sweep_class_bytes / (sweep_ms * 1e-3) * 1e-9 / hbm_peak) if sweep_ms > 0 else None,
        "share_of_step": sweep_ms / (step_ms_spans * args.steps),
        "note": "the local pass (chunk aggregates) reads nothing on the rebuilt rows: it is FP64-pipe work, not traffic",
    }
    if apply_ms >= d_ms or not dense_launches:
        roofline = {
            "bound": "hbm",
            "kernel": "sweep_apply2_kernel (layer sweeps from the true chunk carries, I += I_n, projections of I_n; two columns per thread)",
            "achieved": apply_bytes / (apply_ms * 1e-3) * 1e-9 if apply_ms > 0 else None, "peak": hbm_peak, "unit": "GB/s",
            "frac": (apply_bytes / (apply_ms * 1e-3) * 1e-9 / hbm_peak) if apply_ms > 0 else None,
            "traffic": atr, "traffic_source": anote,
            "algorithmic_bytes_per_element": {"rows with a rebuilt source": 16, "aerosol rows": 32},
            "algorithmic_bytes_per_launch": apply_bytes / max(apply_launches, 1),
            "ms_per_launch": apply_ms / max(apply_launches, 1), "launches": apply_launches,
            "share_of_step": apply_ms / (step_ms_spans * args.steps), "peak_source": hbm_src,
            "timing": "CUDA-event spans on the launching stream in a second pass of the same %d steps (%.2f ms per step with spans; the "
                      "headline pass runs without them, as CUDA-graph replays of two orders each)" % (args.steps, step_ms_spans),
            "sweeps_class": sweeps_class, "contraction": contraction,
        }
    else:
        roofline = dict(contraction, sweeps_class=sweeps_class)

    # ---------------- end to end through the public API (host arrays in, NumPy out) ----------------
    h2d = 0
    d2h = 0
    bs_e2e = sos.BatchSolver(scen, device=dev)

    def step_e2e():
        """What a parameter sweep does per batch: hand the next scenarios (host values) to the resident solver, solve,
        bring the profiles back.  The plan and the phase operands stay (sos_plan_update)."""
        nonlocal h2d, d2h
        bs_e2e.update(scen)                            # host: tau / coefficients of the batch; H2D
        r = bs_e2e.solve(poll_every=2)
        out = bs_e2e.results(r, quadratures=True, fields=False)   # D2H: flux/diffusivity/heating profiles, n, TOA net flux
        # what actually crosses PCIe: tau, the scenario records, and the first-order inputs (table of distinct solar phase
        # vectors + rows + weights: the coefficient planes are assembled on the device, sos_first_order_tab)
        h2d = bs_e2e.tau.nbytes + 80 * len(scen) + bs_e2e.P0tab.nbytes + bs_e2e.P0idx.nbytes + bs_e2e.P0w.nbytes
        d2h = sum(5 * o.flux_up.nbytes for o in out) + 40 * len(out)
        return out

    for _ in range(2):
        step_e2e()
    barrier()
    e2e_times = []
    l1 = bs_e2e.engine.launches
    for k in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        step_e2e()
        torch.cuda.synchronize(dev)
        e2e_times.append(time.perf_counter() - t0)
    e2e_launches = bs_e2e.engine.launches - l1
    te = torch.tensor([float(np.mean(e2e_times))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = units_all / float(te.item())
    bs_e2e.engine.close()

    # the same call with a new plan per batch, and from a cold process state (no cached phase tables / operands / factors)
    def step_new_plan():
        b = sos.BatchSolver(scen, device=dev)
        r = b.solve(poll_every=2)
        b.results(r, quadratures=True, fields=False)
        b.engine.close()

    step_new_plan()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    step_new_plan()
    torch.cuda.synchronize(dev)
    new_plan_ms = 1e3 * (time.perf_counter() - t0)
    sos.clear_caches(disk=False)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    step_new_plan()
    torch.cuda.synchronize(dev)
    cold_ms = 1e3 * (time.perf_counter() - t0)

    # ---------------- the full sweep of BASELINE configs[4]: ~10^4 solves streamed through one resident plan ----------------
    full = None
    if args.full_sweep > 0:
        full = run_full_sweep(args, sos, torch, dist, dev, rank, world, S)

    # ---------------- N > 1: the mu-sharded thick-cloud grid (BASELINE configs[3]) as a secondary record ----------------
    secondary = None
    if world > 1 and args.secondary:
        bs.engine.close()
        del flush
        torch.cuda.empty_cache()
        try:
            rec = thick_record(args, sos, torch, dist, dev, rank, world, 1, 3)
            if rec is not None:
                secondary = {"workload": rec["config"]["workload"], "scaling": "strong", "ms": rec["ms_per_step"], "orders": rec["config"]["orders"],
                             "updates_per_s": rec["value"], "one_gpu_ms": rec.get("one_gpu_ms"), "speedup_vs_1gpu": rec.get("speedup_vs_1gpu"),
                             "sharding": rec["config"]["sharding"], "status": rec["config"]["status"],
                             "bit_identical_to_unsharded": rec.get("bit_identical_to_unsharded")}
        except Exception as e:   # the headline line must not depend on the secondary workload
            secondary = {"workload": "thick FWC cloud layer (BASELINE configs[3])", "error": "%s: %s" % (type(e).__name__, str(e)[:300])}

    if rank == 0:
        line = {
            "metric": "scattering-order updates/s", "value": value, "unit": "updates/s", "n_gpus": world,
            "steps": args.steps, "warmup": W, "ms_per_step": step_ms_max, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(S),
            "details": {"orders_per_scenario": [int(n_orders.min()), int(n_orders.max())], "scenario_orders_per_step": int(np.sum(n_orders - 1)),
                        "l2": "256 MB flush between timed steps; per-step working set %.0f MB > 126 MB L2" % (3 * S * L * eng.ld * 8 / 1e6),
                        "scenarios_swapped_for_blend_overrun": n_swapped,
                        "dealing": ("members 0..%d of the sweep" % (S - 1)) if world == 1 else
                                   ("members 0..%d of the sweep sorted by %s and dealt in serpentine rounds to the %d ranks (every rank a batch "
                                    "of the same make-up; no data-path collective)" % (world * S - 1, dealt_by, world)),
                        "contraction": ("folded (centrosymmetric operands, defect %.1e)" % eng.fold_defect) if folded else "general",
                        "generated_source": generated,
                        "low_rank_operands": [int(r) for r in getattr(eng, "lowrank", [])]},
            "solves_per_s": S * world / (step_ms_max * 1e-3),
            "parity_checked_workload": True,   # tests/test_gpu_workload.py::test_benchmarked_workload_vs_oracle (this batch vs the oracle)
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "updates/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": 1e3 * float(te.item()),
                    "call": "BatchSolver.update(scenarios) + solve() + results(fields=False): host scenario values in, NumPy profiles out, resident plan",
                    "new_plan_per_batch_ms": new_plan_ms, "cold_ms": cold_ms,
                    "cold_note": "cold = first batch of a process: host phase tables (Lorenz-Mie series unless cached on disk), device "
                                 "phase matrices, contraction operands, folded operands, low-rank factors, plan creation, solve, results"},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "wall_s_timed_region": t_wall,
        }
        if full is not None:
            line["full_sweep"] = full
        if per_rank is not None:
            line["per_rank"] = per_rank
        if secondary is not None:
            line["secondary"] = secondary
        if not args.no_cpu and world == 1:   # the CPU baseline leg is an N = 1 item
            units, dt = cpu_port_sample(orders=2)
            line["cpu_baseline"] = {
                "value": units / dt, "unit": "updates/s", "cores": 1, "kind": "port",
                "sample": "1 scenario of the workload, 2 scattering orders at the full 800x1002 grid through the NumPy "
                          "port of the reference algorithm (oracle method='slices', %.1f s); the unmodified reference "
                          "measured 3.0e7 updates/s on one core (BASELINE.md)" % dt}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_full_sweep(args, sos, torch, dist, dev, rank, world, S):
    """BASELINE configs[4] at full size: `args.full_sweep` independent solves (tau_aer x mu0 x omega x albedo x phase
    function), sorted by expected cost (optical depth x single-scattering albedo: the number of orders grows with both) so
    that a batch holds scenarios of similar length, dealt to the ranks batch by batch, and streamed through ONE resident
    plan per rank (BatchSolver.update).  Host work (tau profiles, coefficients, results) is inside the timed region."""
    total = args.full_sweep
    allsc = make_scenarios(sos, total, 0)
    order = sorted(range(total), key=lambda i: -cost_proxy(allsc[i]))
    batches = [order[i:i + S] for i in range(0, total - total % S, S)]          # whole batches only
    mine = batches[rank::world]
    bs = sos.BatchSolver([allsc[i] for i in mine[0]], device=dev)
    n_solves, units, overrun = 0, 0.0, 0
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for b in mine:
        bs.update([allsc[i] for i in b])
        r = bs.solve(poll_every=2)
        try:
            bs.results(r, quadratures=True, fields=False)
        except IndexError:   # a member on which the reference itself raises (blend-search overrun, Q11)
            overrun += int(np.sum((r.status & 1) != 0))
        n_solves += len(b)
        units += float(np.sum(r.n_orders - 1)) * L_DEFAULT * (2 * M_DEFAULT) ** 2
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    t = torch.tensor([dt, float(n_solves), units, float(overrun)], dtype=torch.float64, device=dev)
    if world > 1:
        tm = t.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        dt = float(tm[0].item())
    bs.engine.close()
    return {"solves": int(t[1].item()), "seconds": dt, "solves_per_s": float(t[1].item()) / dt, "updates_per_s": float(t[2].item()) / dt,
            "batch": S, "dealing": "sorted by tau_aer*omega_aer (cost proxy), batches dealt round-robin to the ranks, one resident plan per rank",
            "members_reference_raises_on": int(t[3].item()), "timed": "wall clock over all batches incl. host preparation and D2H of the profiles, max over ranks"}


if __name__ == "__main__":
    main()
