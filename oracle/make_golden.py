"""Generate tests/golden/*.npz by running the UNMODIFIED reference (build container only).

    python oracle/make_golden.py

The reference ships no golden vectors (SURVEY.md §4); these are outputs of the reference
modules themselves (imported through oracle/ref_shims.py from PYLAMP_REFERENCE_DIR) on seeded
inputs.  The inputs are stored next to the outputs so the tests never need the reference.
Test infrastructure only.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shims  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
SEED_C1 = 1234
SEED_THERMO = 4321

# pylamp2.py source-text substitutions for the thermo-mechanical variant (the reference is
# configured by editing the source, README:32-34; only model 5 sets bcstokes, pylamp2.py:239-242)
THERMO_SUBS = [
    ("nx    =   [200+1,40+1] ", "nx    =   [33,49] "),
    ("L     =   [1, 0.2] ", "L     =   [660e3, 1000e3] "),
    ("tracdens = 45 ", "tracdens = 20 "),
    ("tracdens_min = 25 ", "tracdens_min = 0 "),
    ("choose_model = 5", "choose_model = 1"),
    ("bcstokes = [[]] * 4", "bcstokes = [1, 1, 1, 1]"),
]
C1_NOINJECT_SUBS = [("tracdens_min = 25 ", "tracdens_min = 0 ")]
# free-surface stabilisation with the dynamic time step (re-solve loop pylamp2.py:387-405)
C1_SURFSTAB_SUBS = C1_NOINJECT_SUBS + [("surface_stabilization = False ", "surface_stabilization = True ")]


def grids(nx, L):
    grid = [np.linspace(0, L[i], nx[i]) for i in range(2)]
    mesh = np.meshgrid(*grid, indexing="ij")
    gridmp = [(g[1:] + g[:-1]) / 2 for g in grid]
    gridmp = [np.append(g, g[-1] + (g[-1] - g[-2])) for g in gridmp]
    meshmp = np.meshgrid(*gridmp, indexing="ij")
    return grid, mesh, gridmp, meshmp


def kernel_vectors():
    rt, rs, rd, rc = ref_shims.load()
    rng = np.random.default_rng(0)
    out = {}
    nx = [13, 10]
    L = [1.0, 0.7]
    grid, mesh, gridmp, meshmp = grids(nx, L)
    M = 2000
    tr_x = np.clip(rng.random((M, 2)) * L, 1e-3, None)
    f = np.exp(rng.normal(size=(M, 6)))
    out.update(nx=np.array(nx), L=np.array(L), tr_x=tr_x, tr_vals=f)

    # trac2grid on the 4 staggered targets of pylamp2.py:309-313, 319
    sch = [5, 6, 1, 2, 5, 6]
    gf = [np.zeros(nx) for _ in range(6)]
    rt.trac2grid(tr_x, f, mesh, grid, gf, nx, avgscheme=sch)
    out["t2g_nodes_scheme"] = np.array(sch)
    out["t2g_nodes"] = np.array(gf)
    targets = {"cc": ([gridmp[0], gridmp[1]], meshmp),
               "zmid": ([gridmp[0], grid[1]], [meshmp[0], mesh[1]]),
               "xmid": ([grid[0], gridmp[1]], [mesh[0], meshmp[1]])}
    for name, (g, m) in targets.items():
        gf = [np.zeros(nx) for _ in range(2)]
        rt.trac2grid(tr_x, f[:, :2], m, g, gf, nx, avgscheme=[6, 2])
        out["t2g_" + name] = np.array(gf)

    # grid2trac LINEAR / NEAREST, with out-of-grid markers (defval)
    F = [rng.normal(size=nx) for _ in range(2)]
    out["g2t_fields"] = np.array(F)
    xo = tr_x.copy()
    xo[:5, 0] = -0.01
    xo[5:9, 1] = 0.9
    out["g2t_x_outside"] = xo
    for m, name in ((16, "linear"), (8, "nearest")):
        a = np.zeros((M, 2))
        rt.grid2trac(tr_x, a, grid, F, nx, method=m)
        out["g2t_" + name] = a
        a = np.zeros((M, 2))
        import contextlib, io
        with contextlib.redirect_stdout(io.StringIO()):
            rt.grid2trac(xo, a, grid, F, nx, method=m, defval=-7.5)
        out["g2t_" + name + "_outside"] = a

    # cell-centred velocities with BC ring (restated inline steps pylamp2.py:491-545 are
    # exercised by the driver runs below); VELDIV + RK on a ring-padded field
    newvel = [rng.normal(size=nx) * 1e-3 for _ in range(2)]
    velsmp = [0.5 * (newvel[0][1:, :-1] + newvel[0][:-1, :-1]), 0.5 * (newvel[1][:-1, 1:] + newvel[1][:-1, :-1])]
    vels = [np.zeros((nx[0] + 1, nx[1] + 1)) for _ in range(2)]
    for d in range(2):
        vels[d][1:-1, 1:-1] = velsmp[d]
    vels[1][0, :], vels[0][0, :] = vels[1][1, :], -vels[0][1, :]
    vels[0][:, 0], vels[1][:, 0] = vels[0][:, 1], -vels[1][:, 1]
    vels[1][-1, :], vels[0][-1, :] = vels[1][-2, :], -vels[0][-2, :]
    vels[0][:, -1], vels[1][:, -1] = vels[0][:, -2], -vels[1][:, -2]
    ng = [np.insert(gridmp[d], 0, gridmp[d][0] - (gridmp[d][1] - gridmp[d][0])) for d in range(2)]
    out["rk_newvel"] = np.array(newvel)
    out["rk_vels"] = np.array(vels)
    out["rk_grid_z"], out["rk_grid_x"] = ng
    a = np.zeros((M, 2))
    rt.grid2trac(tr_x, a, ng, vels, [nx[0] + 1, nx[1] + 1], defval=0, method=32)
    out["g2t_veldiv"] = a
    out["rk_tstep"] = 0.3
    v, x = rt.RK(tr_x, ng, vels, nx, 0.3)
    out["rk_vel"], out["rk_x"] = v, x

    # Stokes assembly on a non-uniform grid, all usable BC combos, +- surfstab
    gz = np.cumsum(np.r_[0, rng.uniform(0.5, 1.5, nx[0] - 1)])
    gx = np.cumsum(np.r_[0, rng.uniform(0.5, 1.5, nx[1] - 1)])
    g2 = [gz, gx]
    etas = 10 ** rng.uniform(0, 3, nx)
    etan = 10 ** rng.uniform(0, 3, nx)
    rho = rng.uniform(1000, 3000, nx)
    out.update(st_gz=gz, st_gx=gx, st_etas=etas, st_etan=etan, st_rho=rho)
    combos = [[1, 1, 1, 1], [0, 1, 1, 1], [0, 1, 0, 1], [1, 1, 0, 1]]
    out["st_bc"] = np.array(combos)
    for ic, bc in enumerate(combos):
        for ss in (0, 1):
            A, r = rs.makeStokesMatrix(nx, g2, etas, etan, rho, bc, surfstab=bool(ss), tstep=1e3 if ss else None)
            A = A.tocoo()
            key = "st_%d_%d_" % (ic, ss)
            out[key + "row"], out[key + "col"], out[key + "val"], out[key + "rhs"] = A.row, A.col, A.data, r
    # uniform grid too (what the driver uses)
    A, r = rs.makeStokesMatrix(nx, grid, etas, etan, rho, [1, 1, 1, 1])
    A = A.tocoo()
    out["stu_row"], out["stu_col"], out["stu_val"], out["stu_rhs"] = A.row, A.col, A.data, r

    # energy assembly
    gm2 = [(g[1:] + g[:-1]) / 2 for g in g2]
    gm2 = [np.append(g, g[-1] + (g[-1] - g[-2])) for g in gm2]
    T = rng.uniform(300, 1600, nx)
    k = [rng.uniform(1, 5, nx) for _ in range(2)]
    Cp = rng.uniform(800, 1300, nx)
    H = rng.uniform(0, 1e-6, nx)
    out.update(df_T=T, df_k=np.array(k), df_Cp=Cp, df_H=H, df_gmz=gm2[0], df_gmx=gm2[1])
    dcombos = [[0, 1, 0, 1], [1, 0, 1, 0], [0, 0, 0, 0], [1, 1, 1, 1]]
    out["df_bc"] = np.array(dcombos)
    out["df_bcval"] = np.array([273, 1.5, 1623, -2.0])
    out["df_tstep"] = 1e3
    for ic, bc in enumerate(dcombos):
        A, r = rd.makeDiffusionMatrix(nx, g2, gm2, T, k, Cp, rho, H, bc, [273, 1.5, 1623, -2.0], 1e3)
        A = A.tocoo()
        key = "df_%d_" % ic
        out[key + "row"], out[key + "col"], out[key + "val"], out[key + "rhs"] = A.row, A.col, A.data, r
    np.savez_compressed(os.path.join(OUT, "kernels.npz"), **out)
    print("kernels.npz:", len(out), "arrays")


def fence_delete_vectors():
    """The driver-inline fence / delete block (pylamp2.py:557-581) executed as it stands: the lines
    are read from the reference checkout at generation time, dedented and run on crafted markers
    (some beyond every wall), with the fence enabled and disabled."""
    import textwrap
    rt, rs, rd, rc = ref_shims.load()
    lines = open(os.path.join(ref_shims.REFERENCE_DIR, "pylamp2.py")).read().split("\n")
    assert "do not allow tracers to advect outside the domain" in lines[556] and "ntrac = ntrac - dntrac" in lines[580]
    block = compile(textwrap.dedent("\n".join(lines[556:581])), "pylamp2.py:557-581", "exec")
    rng = np.random.default_rng(17)
    L = [1.0, 0.5]
    M = 400
    tr_x0 = (rng.random((M, 2)) * 1.3 - 0.15) * L
    tr_x0[:4] = [[0.0, 0.1], [1.0, 0.2], [0.3, 0.0], [0.4, 0.5]]        # exactly on the walls
    tr_f0 = rng.random((M, rc.NFTRAC))
    tr_f0[:, rc.TR__ID] = np.arange(M)
    vel0 = rng.random((M, 2))
    out = {"fd_L": np.array(L), "fd_tr_x": tr_x0, "fd_tr_f": tr_f0, "fd_vel": vel0}
    for tag, enabled in (("on", True), ("off", False)):
        ns = {"np": np, "DIM": rc.DIM, "IX": rc.IX, "IZ": rc.IZ, "EPS": rc.EPS, "TR__ID": rc.TR__ID, "L": L,
              "pylamp_stokes": rs, "bcstokes": [1, 1, 1, 1], "tracs_fence_enabled": enabled,
              "tr_x": tr_x0.copy(), "tr_f": tr_f0.copy(), "trac_vel": vel0.copy(), "ntrac": M,
              "pprint": lambda *a: None}
        exec(block, ns)
        out["fd_%s_tr_x" % tag], out["fd_%s_tr_f" % tag] = ns["tr_x"], ns["tr_f"]
        out["fd_%s_vel" % tag], out["fd_%s_ntrac" % tag] = ns["trac_vel"], ns["ntrac"]
    np.savez_compressed(os.path.join(OUT, "fence_delete.npz"), **out)
    print("fence_delete.npz: kept", int(out["fd_on_ntrac"]), "(fence on),", int(out["fd_off_ntrac"]), "(fence off) of", M)


def driver_run(name, nsteps, seed, subs, stride):
    cap = ref_shims.run_driver(nsteps, seed, substitutions=subs)
    out = {"seed": seed, "nsteps": nsteps, "stride": stride}
    for it, (g, t) in enumerate(cap):
        for k in ("velz", "velx", "pres", "rho", "temp", "time"):
            out["s%d_%s" % (it, k)] = g[k]
        out["s%d_ntrac" % it] = t["tr_x"].shape[0]
        out["s%d_tr_x" % it] = t["tr_x"][::stride]
        out["s%d_tr_v" % it] = t["tr_v"][::stride]
        out["s%d_tr_T" % it] = t["tr_f"][::stride, 3]
        out["s%d_tr_xsum" % it] = np.sum(t["tr_x"], axis=0)
    out["gridz"], out["gridx"] = cap[0][0]["gridz"], cap[0][0]["gridx"]
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
    print(name, "steps", len(cap), "markers", [int(out["s%d_ntrac" % i]) for i in range(len(cap))])


def flowthru_vectors():
    """Flow-through x = 0 wall (BC_TYPE_FLOWTHRU|FREESLIP = 5, pylamp_stokes.py:268-273, anchor :525-551): the
    reference's matrices on the non-uniform grid of kernels.npz, and its direct solve (spsolve + one refinement
    step) of a 33 x 25 system whose density anomaly next to the wall drives flow through it."""
    import scipy.sparse
    import scipy.sparse.linalg
    rt, rs, rd, rc = ref_shims.load()
    g = np.load(os.path.join(OUT, "kernels.npz"))
    nx = list(g["nx"])
    g2 = [g["st_gz"], g["st_gx"]]
    out = {}
    combos = [[1, 5, 1, 1], [0, 5, 0, 1], [1, 5, 0, 1]]
    out["ft_bc"] = np.array(combos)
    for ic, bc in enumerate(combos):
        A, r = rs.makeStokesMatrix(nx, g2, g["st_etas"], g["st_etan"], g["st_rho"], bc)
        A = A.tocoo()
        key = "ft_%d_" % ic
        out[key + "row"], out[key + "col"], out[key + "val"], out[key + "rhs"] = A.row, A.col, A.data, r
    rng = np.random.default_rng(3)
    nx2, L2 = [33, 25], [1.0, 0.75]
    grid = [np.linspace(0, L2[i], nx2[i]) for i in range(2)]
    z, x = np.meshgrid(grid[0], grid[1], indexing="ij")
    etas = 10 ** (1.5 * np.sin(3 * z) * np.cos(4 * x) + 0.2 * rng.normal(size=nx2))
    etan = 10 ** (1.5 * np.sin(3 * (z + 0.5 / 32)) * np.cos(4 * (x + 0.375 / 24)) + 0.2 * rng.normal(size=nx2))
    rho = 3000 + 200 * np.exp(-((z - 0.4) ** 2 + (x - 0.1) ** 2) / 0.02) + 20 * rng.normal(size=nx2)
    A, r = rs.makeStokesMatrix(nx2, grid, etas, etan, rho, [1, 5, 1, 1])
    A = scipy.sparse.csc_matrix(A)
    lu = scipy.sparse.linalg.splu(A)
    xs = lu.solve(r)
    xs = xs + lu.solve(r - A @ xs)
    out.update(fs_nx=np.array(nx2), fs_gz=grid[0], fs_gx=grid[1], fs_etas=etas, fs_etan=etan, fs_rho=rho, fs_x=xs,
               fs_res=np.linalg.norm(r - A @ xs) / np.linalg.norm(r))
    np.savez_compressed(os.path.join(OUT, "flowthru.npz"), **out)
    vx = xs[1::3].reshape(nx2)
    print("flowthru: residual %.1e, max |vx| on the x = 0 wall %.3e (of %.3e), P(anchor) %.1e" %
          (out["fs_res"], np.abs(vx[:, 0]).max(), np.abs(xs[0::3]).max(), xs[2::3].reshape(nx2)[nx2[0] // 2, 0]))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if "--only-flowthru" in sys.argv:
        flowthru_vectors()
        sys.exit(0)
    if "--only-fence-delete" in sys.argv:
        fence_delete_vectors()
        sys.exit(0)
    if "--only-surfstab" in sys.argv:
        driver_run("c1_surfstab", 3, SEED_C1, C1_SURFSTAB_SUBS, 997)
        sys.exit(0)
    kernel_vectors()
    fence_delete_vectors()
    driver_run("c1_shipped", 3, SEED_C1, [], 997)
    driver_run("c1_noinject", 3, SEED_C1, C1_NOINJECT_SUBS, 997)
    driver_run("thermo_variant", 4, SEED_THERMO, THERMO_SUBS, 53)
    driver_run("c1_surfstab", 3, SEED_C1, C1_SURFSTAB_SUBS, 997)
    flowthru_vectors()
