"""Device-resident thin driver: one pass of the reference's loop body (pylamp2.py:273-594) built
from the same module-level functions pylamp2.py calls, with all state kept in HBM.

Multi-GPU (one process per GPU, `ctx.init_comm()`): the grids are replicated, every rank owns a
share of the markers (trac2grid sums the node sums with an NCCL all-reduce inside the library) and
the Stokes solve is z-slab distributed (halo rows + all-reduced dot products); see DESIGN.md §7.

The unmodified reference driver can also be run against the drop-in modules (INTEGRATION.md), but
its inline NumPy steps then bounce every marker through host memory each call; this driver keeps
markers (SoA columns) and grid fields on the GPU and is what `bench.py` times.

Mirrors oracle/pylamp_oracle.py's State/Options/timestep so that the parity tests read the same on
both sides.  Marker injection (`tracdens_min > 0`), marker removal (`tracs_fence_enabled=False`) and the
`.npz` output (`save_npz`, read back by `load_npz`) are the SURVEY.md §8f rows built so far.
"""
import numpy as np
import torch

from . import _lib, markers, migrate, pylamp_diff, pylamp_stokes, pylamp_trac
from .pylamp_const import *  # noqa: F401,F403
from .pylamp_const import (DIM, EPS, IX, IZ, NFTRAC, SECINYR, TR_ACE, TR_ALP, TR_ET0, TR_ETA, TR_HCD,
                           TR_HCP, TR_IHT, TR_MAT, TR_RH0, TR_RHO, TR_TMP)
from .pylamp_trac import (INTERP_AVG_ARITHW, INTERP_AVG_GEOMETRIC, INTERP_AVG_GEOMW,
                          INTERP_METHOD_LINEAR)
from .setups import make_grids


class Options:
    """The configurable locals of pylamp2.py:37-77 (defaults as shipped)."""

    def __init__(self, **kw):
        self.do_stokes = True
        self.do_advect = True
        self.do_heatdiff = True
        self.do_subgrid_heatdiff = True
        self.tstep_adv_max = 50e9 * SECINYR
        self.tstep_adv_min = 50e-9 * SECINYR
        self.tstep_dif_max = 50e9 * SECINYR
        self.tstep_dif_min = 50e-9 * SECINYR
        self.tstep_modifier = 0.67
        self.tdep_rho = True
        self.tdep_eta = True
        self.etamin = 1e17
        self.etamax = 1e23
        self.Tref = 1623
        self.tracs_fence_enabled = True
        self.surface_stabilization = False      # pylamp2.py:71-73
        self.surfstab_theta = 0.5
        self.surfstab_tstep = -1                # negative: the dynamic time step is used (re-solve loop)
        self.bcstokes = [pylamp_stokes.BC_TYPE_FREESLIP] * 4
        self.bcheat = [pylamp_diff.BC_TYPE_FIXTEMP, pylamp_diff.BC_TYPE_FIXFLOW,
                       pylamp_diff.BC_TYPE_FIXTEMP, pylamp_diff.BC_TYPE_FIXFLOW]
        self.bcheatvals = [273, 0, 1623, 0]
        # solver controls (not in the reference: it calls a direct solver)
        self.stokes_rtol = 1e-12
        self.stokes_maxit = 600
        self.stokes_params = {"warm_start": 1}     # start each solve from the previous step's iterate
        self.heat_rtol = 1e-13
        self.heat_extrapolate = True  # heat solve starts from T + the previous step's increment
        self.resort_every = 0         # > 0: re-order the markers by cell every n-th step (device counting sort)
        self.fused_t2g = True         # the step's marker->grid targets in one pass (plb_trac2grid_fused)
        self.fused_rk4_fence = True   # RK4 + fence + per-cell count in one pass (plb_rk4_fence_count)
        self.tracdens, self.tracdens_min = 45, 0   # marker injection (pylamp2.py:594-633); 0 = off
        # several ranks: "index" = every rank keeps the markers it started with (any marker may be
        # processed by any rank); "slab" = rank r owns the markers in its cell rows, markers that
        # cross a slab boundary migrate to the new owner after the fence (migrate.py)
        self.marker_ownership = "index"
        # slab-owned markers only: combine the node sums by a boundary-row exchange with the neighbouring
        # slabs + an all-gather of the finished rows instead of all-reducing every raw plane (slabgrid.py)
        self.slab_reduce = False
        # slab-owned markers only: SLAB-LOCAL GRID FIELDS (the north_star decomposition) -- a rank keeps the node rows
        # of its own z-slab (+ SLAB_HALO rows of each neighbour) of every grid field current and nothing else:
        # trac2grid adds the boundary rows of neighbouring slabs and exchanges halo rows of the results, the solvers
        # coarsen / solve / return their own rows, reductions are all-reduced scalars.  No full-plane collective
        # is left in the step (DESIGN.md 7).  Takes precedence over `slab_reduce`.
        self.slab_local = True
        # migration by the library's kernels + ncclSend/ncclRecv to the two neighbours (csrc/migrate.cu) instead of
        # the torch.distributed all-to-all of migrate.migrate (kept for the CPU/gloo tests of the host logic)
        self.native_migration = True
        for k, v in kw.items():
            if not hasattr(self, k):
                raise AttributeError(k)
            setattr(self, k, v)


SLAB_HALO = 3     # halo rows of slab-local fields (RK4 reaches 0.67 cells beyond a marker's cell on the half-shifted
                  # centre grid; stencils and interpolations need one row)


def _clamp(v, lo, hi):
    return max(min(v, hi), lo)


def slab_rows(s):
    """Node rows [i0, i1) this rank owns with slab-local fields (the rows of the z-slab solvers: an even split of
    the cell rows, the last rank also owns the last node row), or None."""
    return None if s.ctx.slab is None else s.ctx.slab[:2]


def full_field(s, f):
    """The whole (nz, nxx) field on every rank from slab-local pieces (tests, output): own rows summed over ranks."""
    rows = slab_rows(s)
    if rows is None:
        return f
    g = torch.zeros_like(f)
    g[rows[0]:rows[1]] = f[rows[0]:rows[1]]
    return s.ctx.allreduce(g.view(-1)).view(f.shape) if g.is_contiguous() else g


def _gmax(s, v):
    """max over the ranks of a host scalar (slab-local reductions)."""
    if s.ctx.slab is None:
        return v
    t = torch.tensor([float(v)], dtype=torch.float64, device=s.ctx.torch_device)
    return float(s.ctx.allreduce(t, "max").item())


class State:
    """All arrays the reference driver keeps as locals (pylamp2.py:100-127), in HBM.

    ``tr_x`` is (M,2) [z,x] like the reference; marker properties are 13 separate columns
    (``cols[TR_*]``, SoA) instead of the reference's (M,13) ``tr_f``."""

    def __init__(self, nx, L, tr_x, tr_f, device=None):
        self.ctx = _lib.default_context(device)
        dev = self.ctx.torch_device
        self.nx, self.L = [int(n) for n in nx], [float(v) for v in L]
        self.dx = [self.L[i] / (self.nx[i] - 1) for i in range(DIM)]
        self.grid, self.gridmp = make_grids(self.nx, self.L)
        self.tr_x = _to_dev(tr_x, dev)
        if isinstance(tr_f, (list, tuple)):
            self.cols = [_to_dev(c, dev) for c in tr_f]
        else:
            tf = np.asarray(tr_f)
            self.cols = [_to_dev(np.ascontiguousarray(tf[:, k]), dev) for k in range(NFTRAC)]
        z = lambda: torch.zeros(tuple(self.nx), dtype=torch.float64, device=dev)
        self.f_etas, self.f_T, self.f_rho, self.f_Cp, self.f_etan = z(), z(), z(), z(), z()
        self.f_k = [z(), z()]
        self.f_H, self.f_mat, self.f_sgc = z(), z(), z()
        self.it, self.totaltime = 0, 0.0
        self.newvel, self.newpres, self.newtemp = None, None, None
        self.trac_vel, self.tstep, self.limiter = None, None, ""
        self.kelem, self.count = None, None
        self.stokes_op, self.diff_op = None, None
        self.prev_dT = None
        self.stats = {}

    @property
    def ntrac(self):
        return self.tr_x.shape[0]

    def tr_f_host(self):
        """(M,13) NumPy array in the reference's tr_f layout."""
        return np.stack([c.cpu().numpy() for c in self.cols], axis=1)


def _to_dev(a, dev):
    if isinstance(a, torch.Tensor):
        return a.to(device=dev, dtype=torch.float64).contiguous()
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(dev)


class _Phases:
    """Optional per-phase timing with CUDA events on the current stream (no extra synchronisation:
    the events are resolved by the caller after the step)."""

    def __init__(self, on):
        self.on, self.marks = on, []

    def mark(self, name):
        if self.on:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.marks.append((name, ev))

    def result(self):
        torch.cuda.synchronize()
        out = {}
        for (n0, e0), (n1, e1) in zip(self.marks[:-1], self.marks[1:]):
            out[n1] = out.get(n1, 0.0) + e0.elapsed_time(e1)
        return out


def timestep(s, o, want_kelem=True, phases=False):
    """One pass of the loop body pylamp2.py:273-594 on device-resident state."""
    ctx = s.ctx
    ph = s.phases = _Phases(phases)
    ph.mark("start")
    s.it += 1
    # (first on the second step: the sort's slot table and spare arrays, kept on the state, exist from the start
    # of a run -- a first sort deep inside a run allocates ~8 GB at 2.7e8 markers, measured +70 ms in that step)
    if o.resort_every and s.it >= 2 and (s.it - 2) % o.resort_every == 0:
        if getattr(s, "sort_ws", None) is None:
            s.sort_ws = {}
        s.tr_x, s.cols, _ = markers.sort_by_cell(s.tr_x, s.cols, s.nx, s.L, consume=True, ws=s.sort_ws)
    nx, grid, gridmp = s.nx, s.grid, s.gridmp
    cols, tr_x = s.cols, s.tr_x
    # marker property update, pylamp2.py:291-303
    markers.update_properties(cols[TR_TMP], cols[TR_RH0], cols[TR_ALP], cols[TR_ACE], cols[TR_ET0],
                              o.tdep_rho, o.tdep_eta, o.Tref, o.etamin, o.etamax,
                              rho_out=cols[TR_RHO], eta_out=cols[TR_ETA])
    ph.mark("properties")
    # markers -> grids, pylamp2.py:307-319
    mm = pylamp_trac.marker_minmax(tr_x, ctx)
    t2g = pylamp_trac.trac2grid_device
    world = ctx.comm_info()[1]
    if world > 1 and o.marker_ownership == "slab" and o.slab_local:
        if ctx.slab is None:
            b = migrate.slab_bounds(nx[IZ] - 1, world)
            r = ctx.comm_info()[0]
            ctx.set_slab(b[r], b[r + 1] + (1 if r == world - 1 else 0), SLAB_HALO)
    elif ctx.slab is not None:
        ctx.set_slab(0, 0)
    rows = slab_rows(s)
    own = (lambda f: f[rows[0]:rows[1]]) if rows is not None else (lambda f: f)
    if rows is not None:
        pass        # plb_trac2grid / plb_trac2grid_fused combine the slabs' boundary rows themselves
    elif o.slab_reduce and o.marker_ownership == "slab" and ctx.comm_info()[1] > 1:
        slab_bounds = migrate.slab_bounds(nx[IZ] - 1, ctx.comm_info()[1])

        def t2g(ctx_, x_, cols_, schemes_, grid_, out_, mm_):
            return pylamp_trac.trac2grid_slab(ctx_, x_, cols_, schemes_, grid_, out_, mm_, slab_bounds)
    fused = o.fused_t2g and t2g is pylamp_trac.trac2grid_device
    if o.do_advect and o.do_heatdiff:
        node_cols = [cols[k] for k in (TR_RHO, TR_ETA, TR_HCP, TR_TMP, TR_IHT, TR_MAT)]
        node_sch = [INTERP_AVG_ARITHW, INTERP_AVG_GEOMW] + [INTERP_AVG_ARITHW] * 4
        node_out = [s.f_rho, s.f_etas, s.f_Cp, s.f_T, s.f_H, s.f_mat]
        if not (fused and pylamp_trac.trac2grid_fused_device(
                ctx, tr_x, [(0, node_cols, node_sch, node_out), (1, [cols[TR_ETA]], [INTERP_AVG_GEOMW], [s.f_etan]),
                            (2, [cols[TR_HCD]], [INTERP_AVG_ARITHW], [s.f_k[IZ]]),
                            (3, [cols[TR_HCD]], [INTERP_AVG_ARITHW], [s.f_k[IX]])], grid, gridmp, mm)):
            t2g(ctx, tr_x, node_cols, node_sch, grid, node_out, mm)
            t2g(ctx, tr_x, [cols[TR_ETA]], [INTERP_AVG_GEOMW], gridmp, [s.f_etan], mm)
            t2g(ctx, tr_x, [cols[TR_HCD]], [INTERP_AVG_ARITHW], [gridmp[IZ], grid[IX]], [s.f_k[IZ]], mm)
            t2g(ctx, tr_x, [cols[TR_HCD]], [INTERP_AVG_ARITHW], [grid[IZ], gridmp[IX]], [s.f_k[IX]], mm)
    elif o.do_advect:
        t2g(ctx, tr_x, [cols[TR_RHO], cols[TR_ETA]], [INTERP_AVG_ARITHW, INTERP_AVG_GEOMW], grid,
            [s.f_rho, s.f_etas], mm)
        t2g(ctx, tr_x, [cols[TR_ETA]], [INTERP_AVG_GEOMETRIC], gridmp, [s.f_etan], mm)
    else:
        raise NotImplementedError("heat-only mode (pylamp2.py:321-331) is outside the hot path")
    ph.mark("trac2grid")
    if o.do_heatdiff and s.it > 1:                                                  # :333-337
        s.f_T[:, 0], s.f_T[:, -1] = s.newtemp[:, 0], s.newtemp[:, -1]
        s.f_T[0, :], s.f_T[-1, :] = s.newtemp[0, :], s.newtemp[-1, :]
    if o.do_heatdiff:                                                               # :339-343
        diffusivity = _gmax(s, markers.max_diffusivity2(own(s.f_k[IZ]), own(s.f_rho), own(s.f_Cp)))
        tstep_temp = _clamp(o.tstep_modifier * min(s.dx) ** 2 / diffusivity, o.tstep_dif_min,
                            o.tstep_dif_max)
    ph.mark("dt_heat")
    # Stokes system + solve, pylamp2.py:353-362
    if s.stokes_op is None:
        s.stokes_op = pylamp_stokes.StokesOperator(nx, grid, s.f_etas, s.f_etan, s.f_rho, o.bcstokes,
                                                   ctx=ctx)
        for k, v in o.stokes_params.items():
            s.stokes_op.set_param(k, v)
    else:
        s.stokes_op.set_coeffs(s.f_etas, s.f_etan, s.f_rho)
    if o.surface_stabilization and o.surfstab_tstep >= 0:                           # :354-355
        s.stokes_op.set_surfstab(o.surfstab_tstep, o.surfstab_theta)
    x = s.stokes_op.solve(None, rtol=o.stokes_rtol, maxit=o.stokes_maxit)
    st = s.stokes_op.stats
    s.stats["stokes_iters"] = s.stokes_op.iterations
    s.stats["stokes_relres"] = s.stokes_op.relres
    s.stats["stokes_status"], s.stats["stokes_rtol_eff"], s.stats["stokes_floor"] = st["status"], st["rtol_eff"], st["floor"]
    ph.mark("stokes_solve")
    s.newvel, s.newpres = pylamp_stokes.x2vp(x, nx)
    vmax = _gmax(s, max(markers.field_max(own(s.newvel[IZ])), markers.field_max(own(s.newvel[IX]))))   # :364 (signed)
    tstep_stokes = _clamp(o.tstep_modifier * min(s.dx) / vmax, o.tstep_adv_min, o.tstep_adv_max)
    if o.surfstab_tstep > 0:                                                        # :368-372
        tstep_stokes = o.surfstab_tstep
    if o.do_heatdiff:                                                               # :374-385
        s.limiter = "H" if tstep_temp < tstep_stokes else "S"
        tstep = min(tstep_temp, tstep_stokes)
    else:
        tstep, s.limiter = tstep_stokes, "S"
    if o.surface_stabilization and o.surfstab_tstep < 0:                            # :387-405
        s.stats["stab_solves"] = 0
        while True:      # solve again with the stabilisation terms of the step actually taken
            s.stokes_op.set_surfstab(tstep, o.surfstab_theta)
            x = s.stokes_op.solve(None, rtol=o.stokes_rtol, maxit=o.stokes_maxit)
            s.stats["stab_solves"] += 1
            s.stats["stokes_iters"] += s.stokes_op.iterations
            s.newvel, s.newpres = pylamp_stokes.x2vp(x, nx)
            vmax = _gmax(s, max(markers.field_max(own(s.newvel[IZ])), markers.field_max(own(s.newvel[IX]))))
            check = o.tstep_modifier * min(s.dx) / vmax                            # :399 (not clamped)
            if check < tstep:
                tstep, s.limiter = check, "Ss"
            else:
                break
        ph.mark("stokes_solve")
    s.tstep = tstep
    s.totaltime += tstep
    ph.mark("x2vp_dt")
    if o.do_heatdiff:                                                               # :415-480
        args = (s.f_T, s.f_k, s.f_Cp, s.f_rho, s.f_H, tstep)
        if s.diff_op is None:
            s.diff_op = pylamp_diff.DiffusionOperator(nx, grid, gridmp, *args[:5], o.bcheat,
                                                      o.bcheatvals, tstep, ctx=ctx)
        else:
            s.diff_op.set_coeffs(*args)
        # start from T + the previous step's increment (the increments of consecutive steps are alike)
        guess = s.f_T + s.prev_dT if (o.heat_extrapolate and s.prev_dT is not None) else None
        newtemp = pylamp_diff.x2t(s.diff_op.solve(None, rtol=o.heat_rtol, guess=guess), nx)
        if o.heat_extrapolate:
            s.prev_dT = newtemp - s.f_T
        s.stats["heat_iters"] = s.diff_op.iterations
        ph.mark("heat_solve")
        T = cols[TR_TMP]
        g2t = pylamp_trac.grid2trac_device
        interp = torch.empty_like(T)
        if s.it == 1:                                                               # :441-447
            nbad = g2t(ctx, tr_x, grid, [newtemp], nx, INTERP_METHOD_LINEAR, float("nan"), [interp])
            if nbad:
                raise Exception("stopOnError in grid2trac")
            T.copy_(interp)
        else:                                                                       # :448-480
            dT_grid = newtemp - s.f_T
            if o.do_subgrid_heatdiff:
                # fused: T1 = T + interp(dT_grid); Tsg, dT (:453-475); f_sgc = trac2grid(dT) (:478);
                # T = Tsg - interp(f_sgc) (:479-480)
                Tsg, dT = markers.subgrid_fused(1, tr_x, grid, dT_grid, T, tstep, s.dx[IZ], s.dx[IX],
                                                cols[TR_HCP], cols[TR_RHO], cols[TR_HCD])
                # (one target, one column: the chunk kernel of plb_trac2grid is the faster one here -- measured
                # 0.47 vs 0.77 ms at 2048^2; the fused kernel pays off when several targets share a pass)
                t2g(ctx, tr_x, [dT], [INTERP_AVG_ARITHW], grid, [s.f_sgc], mm)
                markers.subgrid_fused(2, tr_x, grid, s.f_sgc, T, Tsg=Tsg)
            else:
                nbad = g2t(ctx, tr_x, grid, [dT_grid], nx, INTERP_METHOD_LINEAR, float("nan"), [interp])
                if nbad:
                    raise Exception("stopOnError in grid2trac")
                T.add_(interp)
        s.newtemp = newtemp
        ph.mark("grid2trac_T_subgrid")
    # velocities to cell centres + BC ring, RK4, pylamp2.py:491-550
    vzc, vxc = markers.centre_velocities(s.newvel[IZ], s.newvel[IX], o.bcstokes)
    pre = [gridmp[d][0] - (gridmp[d][1] - gridmp[d][0]) for d in range(DIM)]
    newgrid = [np.insert(gridmp[IZ], 0, pre[IZ]), np.insert(gridmp[IX], 0, pre[IX])]
    slab = world > 1 and o.marker_ownership == "slab"
    need_kelem = want_kelem or o.tracdens_min > 0
    flowthru = any(int(b) & pylamp_stokes.BC_TYPE_FLOWTHRU for b in o.bcstokes)
    # (plb_rk4_fence_count: RK4, fence and per-cell count in one pass -- 8.0 vs 7.2 + 1.5 ms at 2.7e8 markers)
    fused_fence = o.fused_rk4_fence and o.tracs_fence_enabled and not slab and not flowthru
    if fused_fence:
        # RK4, fence and per-cell count in one pass over the markers (the new positions are final there)
        s.trac_vel, s.tr_x, s.kelem, s.count = pylamp_trac.rk4_fence_count_device(
            ctx, tr_x, newgrid, vzc, vxc, [nx[IZ] + 1, nx[IX] + 1], tstep, nx, s.L, EPS, want_kelem=need_kelem)
    else:
        s.trac_vel, s.tr_x = pylamp_trac.rk4_device(ctx, tr_x, newgrid, vzc, vxc, [nx[IZ] + 1, nx[IX] + 1], tstep,
                                                    spare=slab)
    ph.mark("advect_rk4")
    # fence (or removal of the markers that left the box) + per-cell count, pylamp2.py:558-593
    if fused_fence:
        pass
    elif not o.tracs_fence_enabled or flowthru:
        if o.tracs_fence_enabled:
            markers.fence(s.tr_x, s.L, EPS, bc=o.bcstokes)                          # every wall but the flow-through ones
        s.stats["removed"] = markers.delete_outside(s)                              # :563-581
        if slab:
            s.stats["migrated"] = (migrate.migrate_native if o.native_migration else migrate.migrate)(s)
        s.kelem, s.count = markers.cell_index_count(s.tr_x, nx, s.L, want_kelem=need_kelem)
    elif slab:
        markers.fence(s.tr_x, s.L, EPS)
        # markers that crossed a slab boundary move to their new owner (positions are final here)
        s.stats["migrated"] = (migrate.migrate_native if o.native_migration else migrate.migrate)(s)
        ph.mark("migrate")
        s.kelem, s.count = markers.cell_index_count(s.tr_x, nx, s.L, want_kelem=need_kelem)
    else:
        s.kelem, s.count = markers.fence_count(s.tr_x, nx, s.L, EPS, want_kelem=need_kelem)
    if o.tracdens_min > 0:                                                          # :594-633
        if world > 1 and not slab:
            raise NotImplementedError("marker injection needs marker_ownership='slab' on several ranks "
                                      "(a cell's markers must live on one rank)")
        cell_rows = None
        if slab:
            # a slab owns every marker of its cell rows: the local counts of those rows are complete
            b = migrate.slab_bounds(nx[IZ] - 1, world)
            cell_rows = (b[ctx.comm_info()[0]], b[ctx.comm_info()[0] + 1])
        s.stats["injected"] = markers.inject_markers(s, o.tracdens, o.tracdens_min, cell_rows=cell_rows)
    if world > 1 and rows is None:
        # per-cell counts of the whole cloud (slab-local fields: every rank keeps the counts of its own cells)
        import torch.distributed as dist
        dist.all_reduce(s.count)
    ph.mark("fence_count")
    return s


def save_npz(s, prefix, it=None):
    """Write the two per-step `.npz` files of the reference with its exact keys (pylamp2.py:637-650:
    `griddata.<it>.npz` = gridz, gridx, velz, velx, pres, rho, temp, tstep, time; `tracs.<it>.npz` =
    tr_x, tr_f, tr_v), so that the reference's pylamp_post.py reads them unchanged (SURVEY.md 8f-2).  On several
    ranks a collective call: rank 0 writes the whole state of every rank (output.write_snapshot)."""
    from .output import write_snapshot
    write_snapshot(s, prefix, it)


def load_npz(prefix, it, o, device=None):
    """The state of a `save_npz` pair (or of the reference's own `griddata.<it>.npz` / `tracs.<it>.npz`), ready for
    `timestep(s, o)`: a collective call on several ranks, where `o.marker_ownership` decides which markers each rank
    keeps (output.read_snapshot)."""
    from .output import read_snapshot
    return read_snapshot(prefix, it, o, device)
