#!/usr/bin/env python
"""bench.py -- PyLamp hot-path benchmark on B200 (one timestep = one pass of the loop body
pylamp2.py:273-594: marker->grid, Stokes solve, energy solve, grid->marker, RK4 advection, fence,
per-cell count).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
  python bench.py --impl reference [--steps K] [--warmup W]      # the reference algorithm on the host CPU
  python bench.py --gpus 1 [...] --dump-outputs DIR               # also write the last timed step's outputs (dump_outputs)

Workload (BASELINE.json configs[3], the one the metric is quoted on): 2-D thermal convection,
Ra=1e6, Arrhenius viscosity clipped to [1e17,1e23], 4096^2 cells (4097^2 nodes), 16 markers/cell
(2.7e8 markers), coupled Stokes + energy + marker advection, synthetic fields generated in HBM.
Prints ONE JSON line (contract in the task statement).  `value` times the device-resident driver;
`e2e` times the same step through host buffers (pinned host -> device marker/field upload and
device -> host result download inside the timed region).  The CPU arm (`--impl reference`, `cpu_baseline`) times a
bounded sample of the same workload (256^2 cells) and scales it to the workload's unit in proportion to the cell count
(`cpu_sample_scaled`: a lower bound on the CPU time; the measured sample numbers are in the same object).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CLASS_NAMES = {0: "k_cheb (Chebyshev-Jacobi smoother sweep, finest level)",
               1: "k_stokes_op (coupled Stokes residual/apply)", 2: "k_multi_dot", 3: "k_multi_axpy2",
               4: "k_t2g_fused + k_t2g_chunk (marker->grid sums: the step's 4-target pass + the subgrid call)", 5: "k_rk4", 6: "k_grid2trac",
               7: "coarse part of the V-cycle (levels >= 1, many launches)",
               8: "finest-level residual+restrict+prolong", 9: "k_precond_rhs", 10: "k_diff", 11: "marker misc",
               12: "k_permute (marker-by-cell sort, when due)"}


def class_name(k):
    return CLASS_NAMES.get(k, "kernel class %d" % k)
SINGLE_KERNEL_CLASSES = (0, 1, 2, 3, 4, 5, 6, 9)


# Solver settings of the timed loop.  stokes_rtol: the scaled TRUE residual (relative to the flow-driving load)
# every timed solve must reach; measured on the B200 (profiles/r02_SUMMARY.md): the fp64 floor of that residual
# at 4097^2 nodes is 2.0e-10 (3e-12 at 513^2), and a solve stopped at 9e-10 is 5e-12 / 1.4e-11 / 9e-15 away from
# the reference's direct solve in vz / vx / P~ (513^2; north_star asks for 1e-8).  tests/test_stokes_large_gpu.py imports exactly these to hold the
# time-loop solver (not a specially tightened one) to the 1e-8 parity bound against the reference's direct
# solve at 513^2 and 1025^2 nodes.
DEFAULTS = {"warm_start": 5, "nu": 2, "gmres_m": 30, "lmax_every": 8, "stokes_rtol": 1e-9, "heat_rtol": 1e-11,
            "resort_every": 16}


def stokes_params(warm_start=None, nu=None, gmres_m=None):
    d = DEFAULTS
    return {"warm_start": d["warm_start"] if warm_start is None else warm_start,
            "gcr_m": d["gmres_m"] if gmres_m is None else gmres_m, "lmax_every": d["lmax_every"],
            "nu": d["nu"] if nu is None else nu,
            "graph_all": 0}     # keep the V-cycle's kernels individually event-timed (whole-cycle graph: no gain at 4096^2)


def peaks():
    """HBM peak: MEASURED_PEAKS.json (driver-written) else the profiling guide's fallback."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy bandwidth measured on this pool's B200)"
        except Exception:
            pass
    return 7700.0, "fallback: B200_PROFILING.md nominal HBM3e 7.7 TB/s"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index=0, period=0.05):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.period, self._stop_evt = period, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
                 "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80)}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def workload_name(ncell, per_side):
    return ("C4 thermal convection Ra=1e6, Arrhenius viscosity clipped [1e17,1e23], "
            "%d^2 cells, %d markers/cell, Stokes+energy+MIC advection" % (ncell, per_side ** 2))


def cpu_sample_scaled(sec, sample_ncell, sample_markers, ncell):
    """The CPU path cannot run the workload itself (SuperLU at 4096^2: days, > host RAM), so a time step of a bounded
    SAMPLE of it is timed -- the same setup on sample_ncell^2 cells -- and scaled to the metric's unit, time steps of the
    ncell^2 workload per second, in proportion to the cell count.  Proportional scaling is a LOWER bound on the CPU
    time: the measured law of the direct solve is x12 per doubling of the side (BASELINE.md) / x23 for x4 the cells
    (256^2 -> 512^2, profiles/r02_SUMMARY.md), i.e. super-linear.  Returns (seconds per workload step, factor, text)."""
    factor = (float(ncell) / float(sample_ncell)) ** 2
    text = ("measured: %.3f s per step of the same C4 setup on %d^2 cells (%d markers) = %.4g timesteps/s of the sample, "
            "1 of the host's %d cores (the NumPy/SuperLU path is single-threaded); scaled to the %d^2-cell workload in "
            "proportion to the cell count (x%.0f): a lower bound on the CPU time -- SuperLU grows x12 per doubling of "
            "the side (BASELINE.md: 0.15/0.95/11.2/140.6 s per solve at 64^2/128^2/256^2/512^2) and cannot run 4096^2 "
            "(days, > host RAM)" % (sec, sample_ncell, sample_markers, 1.0 / sec, os.cpu_count() or 0, ncell, factor))
    return sec * factor, factor, text


def cpu_reference_steps(ncell, nsteps, warmup):
    """The reference algorithm (oracle restatement of pylamp2.py's loop body with scipy spsolve)
    on the host CPU: returns (seconds per step list, nx, markers, per-phase timers)."""
    from oracle import pylamp_oracle as O
    from pylamp_b200 import setups
    nx, L, tr_x, tr_f, opts = setups.convection(ncell=ncell)
    s, o = O.State(nx, L, tr_x, tr_f), O.Options(**opts)
    times, timers = [], {}
    for it in range(warmup + nsteps):
        t = time.perf_counter()
        O.timestep(s, o, timers if it >= warmup else None)
        if it >= warmup:
            times.append(time.perf_counter() - t)
    return times, nx, tr_x.shape[0], timers


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncell = args.ref_ncell
    times, nx, M, timers = cpu_reference_steps(ncell, args.steps, args.warmup)
    sec_sample = float(np.mean(times))
    sec, factor, sample = cpu_sample_scaled(sec_sample, ncell, M, args.ncell)
    cores = 1
    W = args.ncell
    line = {"impl": "reference", "metric": "timesteps_per_s", "value": 1.0 / sec, "unit": "timesteps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            # the workload of the GPU arm; what was actually run is the bounded sample described in cpu_baseline
            "config": {"workload": workload_name(W, args.per_side), "grid_nodes": [W + 1, W + 1],
                       "markers": W * W * args.per_side ** 2, "stokes_dof": 3 * (W + 1) * (W + 1),
                       "sample_grid_nodes": nx, "sample_markers": M, "sample_scale_factor": factor},
            "stokes_dof_per_s": 3.0 * nx[0] * nx[1] / sec_sample,          # measured on the sample (size-independent unit)
            "cpu_baseline": {"value": 1.0 / sec, "unit": "timesteps/s", "cores": cores, "host_cores": os.cpu_count(),
                             "kind": "port", "sample": sample, "sample_timesteps_per_s": 1.0 / sec_sample,
                             "sample_ms_per_step": sec_sample * 1e3, "scale_factor": factor,
                             "phases_s": {k: v / args.steps for k, v in timers.items()}},
            "e2e": {"value": 1.0 / sec, "unit": "timesteps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs one GPU (on several the markers and grid rows are split over the ranks)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from pylamp_b200 import _lib, driver, setups
    ctx = _lib.default_context(local)
    if world > 1:
        ctx.init_comm()           # NCCL communicator of the slab solver / marker-parallel trac2grid
    ncell = args.ncell
    nx, L, tr_x, cols, opts = setups.convection_device(ncell=ncell, per_side=args.per_side, seed=args.seed,
                                                       device="cuda:%d" % local, rank=rank, world=world)
    s = driver.State(nx, L, tr_x, cols, device=local)
    o = driver.Options(**opts)
    o.heat_rtol = args.heat_rtol
    o.marker_ownership = args.marker_ownership
    o.slab_reduce = bool(args.slab_reduce)
    o.slab_local = bool(args.slab_local)
    o.resort_every = args.resort_every
    o.fused_rk4_fence = bool(args.fused_rk4_fence)
    o.stokes_rtol = args.stokes_rtol
    o.stokes_params = stokes_params(args.warm_start, args.nu, args.gmres_m)
    M = s.ntrac
    if world > 1:
        tm = torch.tensor([M], dtype=torch.int64, device="cuda")
        dist.all_reduce(tm)
        M = int(tm.item())
    N = nx[0] * nx[1]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # spin-up (part of the workload set-up, untimed): the synthetic initial state relaxes for a few
    # steps (marker temperatures settle on the grid solution, the flow field develops) before the
    # warm-up and the timed steps run on a smoothly evolving state
    for _ in range(args.spinup + args.warmup):
        driver.timestep(s, o, want_kelem=False)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ctx.profile(True)
    l0 = ctx.launches
    prof = {}
    iters = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    phase_ms, step_ms, step_rk4 = {}, [], []
    for _ in range(args.steps):
        driver.timestep(s, o, want_kelem=False, phases=True)
        iters.append(dict(s.stats))
        pr = s.phases.result()
        step_ms.append(round(sum(pr.values()), 2))
        step_rk4.append(round(pr.get("advect_rk4", 0.0), 2))
        for k, v in pr.items():
            phase_ms[k] = phase_ms.get(k, 0.0) + v / args.steps
        for k, (c, ms, by) in ctx.profile_read().items():
            a = prof.setdefault(k, [0, 0.0, 0.0])
            a[0] += c
            a[1] += ms
            a[2] += by
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    ctx.profile(False)
    launches = ctx.launches - l0
    clocks = sampler.stop()
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    if args.dump_outputs:                        # before the e2e leg moves the state on
        dump_outputs(s, args.per_side, args.dump_outputs)

    # ---- e2e: the same step through host buffers (rank-local) ----
    e2e = None
    if args.e2e_steps > 0:
        e2e = run_e2e(torch, driver, s, o, args.e2e_steps)
        if world > 1:                            # time: the slowest rank; bytes: the whole job's
            t = torch.tensor([e2e["ms"]], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e["ms"] = float(t.item())
            b = torch.tensor([e2e["h2d"], e2e["d2h"]], dtype=torch.float64, device="cuda")
            dist.all_reduce(b, op=dist.ReduceOp.SUM)
            e2e["h2d"], e2e["d2h"] = int(b[0].item()), int(b[1].item())

    if world > 1:
        # nothing collective happens after this point: the other ranks must not wait for rank 0's report
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peak, peak_src = peaks()
    single = {k: v for k, v in prof.items() if k in SINGLE_KERNEL_CLASSES}
    dom = max(single, key=lambda k: single[k][1]) if single else None
    roofline = None
    if dom is not None:
        c, ms, by = prof[dom]
        ach = by / (ms * 1e-3) / 1e9
        traffic = None
        try:        # DRAM bytes per launch from the committed ncu --set full capture (same kernel, same grid)
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            key = {0: "k_cheb", 4: "k_t2g"}.get(dom)
            if key and tr[key]["grid_nodes"] == list(nx) and world == 1:
                traffic = tr[key]["dram_bytes_per_launch"]
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": class_name(dom), "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": ach / peak, "traffic": traffic, "launches_timed": c, "avg_launch_ms": ms / c,
                    "algorithmic_bytes_per_launch": by / c, "peak_source": peak_src,
                    "share_of_step": ms / (ms_step * args.steps)}
    # the stencil/smoother kernel (north_star's ">= 60 % of HBM roofline in the stencil/smoother kernels")
    roofline_stencil = None
    if 0 in prof and prof[0][1] > 0:
        c, ms, by = prof[0]
        ach = by / (ms * 1e-3) / 1e9
        roofline_stencil = {"bound": "hbm", "kernel": class_name(0), "achieved": ach, "peak": peak, "unit": "GB/s",
                            "frac": ach / peak, "avg_launch_ms": ms / c, "share_of_step": ms / (ms_step * args.steps)}
    breakdown = {class_name(k): {"launch_groups": v[0], "ms_per_step": v[1] / args.steps,
                                  "GBps": (v[2] / (v[1] * 1e-3) / 1e9) if v[1] > 0 and v[2] > 0 else None}
                 for k, v in sorted(prof.items())}
    value = 1.0 / (ms_step * 1e-3)            # ONE global problem on all ranks (strong scaling)
    line = {"metric": "timesteps_per_s", "value": value, "unit": "timesteps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(ncell, args.per_side),
                       "grid_nodes": nx, "markers": M, "stokes_dof": 3 * N,
                       "parallelism": "1 GPU" if world == 1 else
                       "%d GPUs, one problem in z-slabs: %s" %
                       (world, "slab-owned markers that migrate after every step, slab-local grid fields (boundary-row "
                        "accumulate + halo rows over NCCL send/recv, all-reduced scalars; no full-plane collective)"
                        if (args.marker_ownership == "slab" and args.slab_local) else
                        ("slab-owned markers with migration, replicated fields" if args.marker_ownership == "slab" else
                         "markers shared by index, replicated fields, raw node sums all-reduced")),
                       "marker_order": "device counting sort by cell every %d steps (inside the timed region when due)" % args.resort_every
                       if args.resort_every else "never re-sorted",
                       "l2_policy": "every field (%.0f MB) and marker array exceeds the 126 MB L2; no flush needed" % (8 * N / 1e6),
                       "spinup_steps": args.spinup, "stokes_rtol": o.stokes_rtol,
                       "stokes_rtol_eff_max": max(i.get("stokes_rtol_eff", 0.0) for i in iters),
                       "stokes_relres_max": max(i.get("stokes_relres", 0.0) for i in iters),
                       "stokes_floor_est_max": max(i.get("stokes_floor", 0.0) for i in iters),
                       "stokes_all_converged_to_rtol": all(i.get("stokes_status") == "converged" for i in iters), "heat_rtol": o.heat_rtol, "smoother_steps": args.nu, "stokes_solver": "FGMRES(%d) + GMG V(nu,nu) Chebyshev-Jacobi (--nu), warm start by polynomial extrapolation of the last %d iterates, eigenvalue estimates every 8 steps" % (args.gmres_m, args.warm_start)},
            "stokes_dof_per_s": 3.0 * N / (ms_step * 1e-3),
            "solver_iterations": iters, "clocks": clocks, "gpu_launches": int(launches),
            "roofline": roofline, "roofline_stencil": roofline_stencil, "phases_ms_per_step": phase_ms,
            "ms_of_each_timed_step": step_ms, "advect_rk4_ms_of_each_timed_step": step_rk4,
            "kernel_breakdown": breakdown}
    if e2e is not None:
        line["e2e"] = {"value": 1.0 / (e2e["ms"] * 1e-3), "unit": "timesteps/s",
                       "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"], "steps": args.e2e_steps}
    if world == 1 and args.cpu_ncell > 0:
        times, cnx, cM, timers = cpu_reference_steps(args.cpu_ncell, 2, 0)
        sec_sample = float(np.mean(times))
        sec, factor, sample = cpu_sample_scaled(sec_sample, args.cpu_ncell, cM, ncell)
        line["cpu_baseline"] = {"value": 1.0 / sec, "unit": "timesteps/s", "cores": 1, "host_cores": os.cpu_count(),
                                "kind": "port", "sample": "2 steps; " + sample,
                                "sample_timesteps_per_s": 1.0 / sec_sample, "sample_ms_per_step": sec_sample * 1e3,
                                "scale_factor": factor,
                                "stokes_dof_per_s": 3.0 * cnx[0] * cnx[1] / sec_sample,
                                "phases_s": {k: v / 2 for k, v in timers.items()}}
    print(json.dumps(line), flush=True)


DUMP_NODES, DUMP_MARKERS, DUMP_SEED, DUMP_MAX_BYTES = 1 << 19, 1 << 18, 2024, 64 * 10 ** 6


def dump_outputs(s, per_side, out_dir):
    """Writes what the last timed step hands back, the arrays of the reference's per-step output (pylamp2.py:637-650,
    driver.save_npz): the grids velz, velx, pres, rho, temp and the markers' tr_x (M,2), tr_f (M,13), tr_v (M,2), as
    out_dir/<name>.npy in float64.  A fixed seeded sample keeps the files under DUMP_MAX_BYTES: DUMP_NODES nodes of
    every grid (flat indices, ascending) and every marker of DUMP_MARKERS / per_side^2 cells, ordered by (cell, z, x)
    -- the device sort orders the markers of one cell by the arrival of its atomics, so the sample is put in an order
    of its own that two runs of one build share.  The cells are those the markers sit in after the last step, and the
    markers carry no identity (the TR__ID column of this workload is zero): where two builds move a marker to
    different sides of a sampled cell's edge, the marker arrays differ in length or shift by a row, so compare two
    builds' markers cell by cell (the cell of a row follows from its tr_x), not row by row.  The grid samples always
    align."""
    import torch
    nz, nxx = s.nx
    dev = s.tr_x.device
    rng = np.random.default_rng(DUMP_SEED)
    nodes = np.sort(rng.choice(nz * nxx, min(nz * nxx, DUMP_NODES), replace=False))
    ncells = (nz - 1) * (nxx - 1)
    cells = rng.choice(ncells, min(ncells, max(1, DUMP_MARKERS // per_side ** 2)), replace=False)
    inode = torch.as_tensor(nodes, device=dev)
    out = {name: f.reshape(-1)[inode].cpu().numpy() for name, f in
           (("velz", s.newvel[0]), ("velx", s.newvel[1]), ("pres", s.newpres), ("rho", s.f_rho), ("temp", s.newtemp))}
    # cell of every marker: floor((n-1)*x/L) clamped into the box, the key of the device sort
    ie = torch.floor((nz - 1) * s.tr_x[:, 0] / s.L[0]).clamp_(0, nz - 2).long()
    key = ie * (nxx - 1) + torch.floor((nxx - 1) * s.tr_x[:, 1] / s.L[1]).clamp_(0, nxx - 2).long()
    del ie
    picked = torch.zeros(ncells, dtype=torch.bool, device=dev)
    picked[torch.as_tensor(cells, device=dev)] = True
    m = torch.nonzero(picked[key]).squeeze(1)
    key = key[m].cpu().numpy()
    x = s.tr_x[m].cpu().numpy()
    m = m[torch.as_tensor(np.lexsort((x[:, 1], x[:, 0], key)), device=dev)]
    out["tr_x"] = s.tr_x[m].cpu().numpy()
    out["tr_f"] = torch.stack([c[m] for c in s.cols], dim=1).cpu().numpy()
    out["tr_v"] = s.trac_vel[m].cpu().numpy()
    nbytes = sum(a.nbytes for a in out.values())
    if nbytes > DUMP_MAX_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (nbytes, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def run_e2e(torch, driver, s, o, nsteps):
    """The same timestep through HOST buffers.  What a time step takes in and hands back is the state that changes:
    marker coordinates and marker temperature go from pinned host memory to the device, the step runs, and the new
    coordinates, marker temperature, marker velocities and the velocity / pressure / temperature grids come back
    (the constant material columns -- rho0, alpha, Ea, eta0, k, Cp, H, material id -- are uploaded once with the
    set-up, like the grids' axes; on several GPUs they migrate with their markers on the device).  Step n+1 can only
    start from what step n returned, so upload -> step -> download of (coordinates, temperature) is a serial chain;
    the outputs that are not fed back (marker velocities, grids) are downloaded on a second stream while the next
    step's upload runs (PCIe is full duplex).  Everything is inside the timed region; both streams are drained
    before the clock stops.  With slab-owned markers a rank's marker count changes from step to step: the pinned
    buffers have head-room and every copy moves the rows in use (bytes counted per step from those rows)."""
    from pylamp_b200.pylamp_const import TR_TMP
    M0 = int(s.tr_x.shape[0])
    cap = M0 + M0 // 4 + 1024
    h_x = torch.empty((cap, 2), dtype=torch.float64, pin_memory=True)
    h_T = torch.empty(cap, dtype=torch.float64, pin_memory=True)
    h_v = torch.empty((cap, 2), dtype=torch.float64, pin_memory=True)
    h_x[:M0].copy_(s.tr_x)
    h_T[:M0].copy_(s.cols[TR_TMP])
    h_grids = [torch.empty(tuple(s.nx), dtype=torch.float64, pin_memory=True) for _ in range(4)]
    h2d = d2h = 0
    side = torch.cuda.Stream()
    main = torch.cuda.current_stream()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(nsteps):
        M = int(s.tr_x.shape[0])                 # rows this rank holds (= what the last download wrote)
        s.tr_x.copy_(h_x[:M], non_blocking=True)
        s.cols[TR_TMP].copy_(h_T[:M], non_blocking=True)
        h2d += 3 * M * 8
        driver.timestep(s, o, want_kelem=False)
        M = int(s.tr_x.shape[0])
        if M > cap:
            raise RuntimeError("e2e: a rank's marker count outgrew the host buffers (%d > %d)" % (M, cap))
        done = torch.cuda.Event()
        done.record(main)
        vel = s.trac_vel if (s.trac_vel is not None and s.trac_vel.shape[0] == M) else None
        outs = [(h_grids[0], s.newvel[0]), (h_grids[1], s.newvel[1]), (h_grids[2], s.newpres), (h_grids[3], s.newtemp)]
        if vel is not None:
            outs.append((h_v[:M], vel))
        with torch.cuda.stream(side):
            side.wait_event(done)
            for h, d in outs:
                d.record_stream(side)            # the next step replaces these tensors while the copy may still run
                h.copy_(d, non_blocking=True)
                d2h += d.numel() * 8
        h_x[:M].copy_(s.tr_x, non_blocking=True)
        h_T[:M].copy_(s.cols[TR_TMP], non_blocking=True)
        d2h += 3 * M * 8
        main.synchronize()                       # the next step starts from h_x, h_T
    side.synchronize()
    ev1.record()
    torch.cuda.synchronize()
    return {"ms": ev0.elapsed_time(ev1) / nsteps, "h2d": int(h2d // nsteps), "d2h": int(d2h // nsteps)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--spinup", type=int, default=8, help="untimed set-up steps before the warm-up (developed flow state)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ncell", type=int, default=4096, help="cells per side of the GPU workload")
    ap.add_argument("--per-side", type=int, default=4, help="markers per cell side (16/cell)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--heat-rtol", type=float, default=DEFAULTS["heat_rtol"], help="tolerance of the energy solve")
    ap.add_argument("--stokes-rtol", type=float, default=DEFAULTS["stokes_rtol"],
                    help="tolerance of the Stokes solve (scaled true residual, relative to the flow-driving load)")
    ap.add_argument("--warm-start", type=int, default=DEFAULTS["warm_start"], help="Stokes initial guess: 0 zero, 1 previous iterate, p >= 2: polynomial extrapolation of the last p iterates")
    ap.add_argument("--nu", type=int, default=DEFAULTS["nu"], help="Chebyshev steps per pre-/post-smoothing")
    ap.add_argument("--gmres-m", type=int, default=DEFAULTS["gmres_m"], help="FGMRES restart length of the Stokes solve")
    ap.add_argument("--marker-ownership", default="slab", choices=["index", "slab"],
                    help="several GPUs: markers are owned by z-slab and migrate (slab, default) or stay with their rank (index)")
    ap.add_argument("--slab-local", type=int, default=1,
                    help="with --marker-ownership slab: slab-local grid fields, no full-plane collective (default)")
    ap.add_argument("--slab-reduce", type=int, default=0,
                    help="with --marker-ownership slab --slab-local 0: boundary-row exchange + all-gather instead of the all-reduce")
    ap.add_argument("--resort-every", type=int, default=DEFAULTS["resort_every"],
                    help="re-sort the markers by cell every n-th step (0: never)")
    ap.add_argument("--fused-rk4-fence", type=int, default=1, help="RK4 + fence + per-cell count in one kernel (1 GPU)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="label of the JSON line: 'strong' = the 4096^2 problem on N GPUs (default); 'weak' when --ncell is "
                         "chosen per N so that the work per GPU stays fixed (SURVEY 8d C5: 4096, 5632, 8192, 11264 cells)")
    ap.add_argument("--seed", type=int, default=11, help="seed of the marker jitter (rank r uses seed + 1000 r)")
    ap.add_argument("--cpu-ncell", type=int, default=256, help="CPU-baseline sample size (0 = skip)")
    ap.add_argument("--ref-ncell", type=int, default=256, help="--impl reference sample size")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write a fixed sample of what the last one computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
