/* pylamp_b200.h -- C ABI of libpylamp_b200.so: PyLamp's per-timestep hot path on B200 (sm_100a).
 *
 * The reference (larskaislaniemi/PyLamp) has no FFI: its boundary is the set of module-level
 * Python functions that pylamp2.py calls.  Each entry point below replaces one of them (the
 * reference file:line is cited per function); the Python modules in pylamp_b200/ keep the
 * reference's names and signatures and reach these symbols through ctypes.
 *
 * Conventions
 *   - plain C types only; every `d_` pointer is DEVICE memory, every `h_` pointer HOST memory.
 *   - all floating point is IEEE fp64 (the reference is NumPy float64 throughout).
 *   - grid fields are row-major [i (z)][j (x)], x fastest, with a leading dimension `ld >= nxx`
 *     in doubles (ld == nxx reproduces the reference's C-contiguous layout).
 *   - marker coordinates `d_tr_x` are (M,2) [z,x] pairs exactly like the reference's tr_x;
 *     marker properties are passed as separate columns (SoA), one device pointer per column.
 *   - every function returns 0 on success, non-zero on error; plb_last_error() gives the text.
 *     No exceptions cross the boundary.  Work is enqueued on the context's stream; functions
 *     that return values through `h_` pointers synchronise that stream.
 */
#ifndef PYLAMP_B200_H
#define PYLAMP_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct plb_ctx plb_ctx;
typedef struct plb_stokes plb_stokes;
typedef struct plb_diff plb_diff;

/* averaging schemes and interpolation methods: pylamp_trac.py:11-22 */
#define PLB_AVG_ARITHMETIC 1
#define PLB_AVG_GEOMETRIC 2
#define PLB_AVG_WEIGHTED 4
#define PLB_METHOD_NEAREST 8
#define PLB_METHOD_LINEAR 16
#define PLB_METHOD_VELDIV 32
/* Stokes wall types pylamp_stokes.py:17-20; heat wall types pylamp_diff.py:12-13 */
#define PLB_BC_NOSLIP 0
#define PLB_BC_FREESLIP 1
#define PLB_BC_CYCLIC 2
#define PLB_BC_FLOWTHRU 4
#define PLB_BC_FIXTEMP 0
#define PLB_BC_FIXFLOW 1
#define PLB_MAX_FIELDS 8

/* ---- context ------------------------------------------------------------------------- */
int plb_ctx_create(int device, plb_ctx** out);
void plb_ctx_destroy(plb_ctx* ctx);
/* run on an existing cudaStream_t (e.g. torch's current stream); 0 = CUDA's default stream.
 * A fresh context owns a private non-blocking stream until this is called. */
int plb_ctx_set_stream(plb_ctx* ctx, void* cuda_stream);
int plb_ctx_sync(plb_ctx* ctx);
const char* plb_last_error(plb_ctx* ctx);
/* number of CUDA kernels this library has launched on the context so far */
long long plb_launch_count(plb_ctx* ctx);
/* tuning knobs that never change results beyond summation order.  "t2g_variant": 1 (default) =
 * plb_trac2grid uses the wide-load chunk kernel when every scheme is weighted and the arrays are
 * 32-byte aligned; 2 = the same kernel, additionally combining the chunks' first runs across the
 * lanes of a warp (fewer atomics on staggered targets and displaced clouds); 0 = always the generic
 * scatter kernel. */
int plb_ctx_set_param(plb_ctx* ctx, const char* name, double value);
const char* plb_version(void);
/* per-kernel-class timing with CUDA event pairs recorded around the launches on the context's
 * stream (classes: 0 smoother sweep on the finest level, 1 coupled Stokes operator, 2 multi-dot,
 * 3 multi-axpy, 4 trac2grid scatter, 5 RK4, 6 grid2trac, 7 coarse part of a V-cycle, 8 finest-level
 * residual/restriction/prolongation, 9 preconditioner rhs, 10 heat operator, 11 other marker
 * kernels).  plb_profile_read fills h_count[16], h_ms[16], h_bytes[16] (algorithmic bytes of the
 * recorded launches, DESIGN.md) and resets. */
int plb_profile_enable(plb_ctx* ctx, int on);
int plb_profile_read(plb_ctx* ctx, long long* h_count, double* h_ms, double* h_bytes);

/* ---- multi-GPU: one process per GPU, z-slab decomposition (SURVEY.md 8e) ------------------------
 * Rank 0 creates a 128-byte NCCL unique id, the host side distributes it (e.g. torch.distributed
 * broadcast) and every rank calls plb_comm_init.  Afterwards Stokes operators created on the
 * context are slab-distributed: halo rows travel with grouped ncclSend/ncclRecv, dot products and
 * other small reductions with ncclAllReduce, all on the context's stream.  The reference's own
 * scheme (replicated data + MPI Allreduce of marker-sized arrays, pylamp2.py:446-555) is not reused. */
int plb_comm_unique_id(plb_ctx* ctx, char* h_id128);
int plb_comm_init(plb_ctx* ctx, int rank, int size, const char* h_id128);
int plb_comm_info(plb_ctx* ctx, int* h_rank, int* h_size);
/* in-place all-reduce of a device buffer of doubles; op: 0 sum, 1 max, 2 min */
int plb_allreduce(plb_ctx* ctx, double* d_buf, long long count, int op);
/* Slab-local grid fields (north_star: "the domain shards naturally into slabs"; replaces the replicated data +
 * Allreduce of pylamp2.py:445-455, :550-555).  After plb_ctx_set_slab(i0, i1, halo) the context's rank keeps
 * only the node rows [i0, i1) of every (nz x ld) grid field current -- the rows of its z-slab of the Stokes and
 * heat solvers; the last rank also owns the last node row -- plus `halo` rows of each neighbour, and its markers
 * must lie in the cell rows [i0, min(i1, nz-1)) (pylamp_b200/migrate.py moves them after advection).  Then
 * plb_trac2grid / plb_trac2grid_fused add the boundary rows of neighbouring slabs (grouped ncclSend/ncclRecv),
 * finish the own rows and exchange halo rows of the results instead of all-reducing whole planes;
 * plb_stokes_solve / plb_diff_solve return their own rows plus halo rows (no zero-filled full-size vector to sum).
 * i1 <= i0 switches back to replicated fields.  plb_halo_rows: exchange `h` halo rows of narr full-size arrays
 * (h_row_doubles[a] doubles per row) with both z-neighbours, one NCCL group. */
int plb_ctx_set_slab(plb_ctx* ctx, int i0, int i1, int halo);
/* Removal of the markers beyond the box, pylamp2.py:563-581 (fence disabled, or a flow-through wall: the reference
 * flags them TR__ID = -1 and np.delete's their rows from tr_x, tr_f, trac_vel).  All arrays (coordinates first; rows of
 * 1 or 2 doubles) lose the same rows: survivors of the tail move into the holes -- marker order is free --, *h_M_new
 * rows remain in use. */
int plb_delete_outside(plb_ctx* ctx, long long M, int narr, double* const* h_arrs, const int* h_width, double Lz, double Lx,
                       long long* h_M_new);

/* Marker injection into under-populated cells, pylamp2.py:594-633 (the reference's Python loop with np.append per
 * cell).  plb_inject_plan: among the cells [cell0, cell1) (a slab serves its own rows) those with fewer than
 * tracdens_min markers receive tracdens - count new ones; h_out[3] = {deficient cells, markers to add, sum of
 * (added - 1) = what these cells advance the marker ids by}.  plb_inject_apply appends the planned markers behind the
 * M existing ones (d_tr_x and the ncols distinct columns need room for M + added rows): positions uniformly random
 * inside the cell from a counter-based Philox4x32-10 stream (seed, stream0 + marker number) -- the reference's global
 * Mersenne-Twister stream cannot be reproduced on a device, parity is at the level of counts, cells, properties
 * and ids --, properties = mean of the cell's existing markers (0/0 = NaN for an empty cell, like the reference),
 * ids continuing from id_start exactly as the reference's loop does (each cell's first new id repeats the running
 * maximum, :614-615).  d_kelem / d_count: cell index per marker and markers per cell (plb_cell_index_count). */
int plb_inject_plan(plb_ctx* ctx, long long ncell, const long long* d_count, int tracdens, int tracdens_min,
                    long long cell0, long long cell1, long long* h_out);
int plb_inject_apply(plb_ctx* ctx, long long M, const long long* d_kelem, const long long* d_count, double* d_tr_x,
                     int ncols, double* const* h_cols, int id_col, double id_start, const double* d_grid_z,
                     const double* d_grid_x, int nxx, unsigned long long seed, unsigned long long stream0);

/* Marker migration between z-slabs after advection (north_star; replaces pylamp2.py:550-555's Allreduce of all
 * positions): rank r owns the markers whose cell row floor((nz-1)*z/Lz) (pylamp2.py:588) lies in [c0, c1).
 * plb_migrate_plan lists the leavers (one pass over the coordinates), swaps the counts with the two neighbours
 * and returns h_counts[4] = {leavers down, leavers up, arrivals from below, arrivals from above}; a marker that
 * moved beyond the neighbouring slab is an error (CFL 0.67 allows 0.45 cells per step).  plb_migrate_apply packs
 * the leavers' rows of all arrays (coordinates first; rows of 1 or 2 doubles; capacity_rows rows allocated, M in
 * use), exchanges them with one grouped ncclSend/ncclRecv pair per neighbour, writes the arrivals into the
 * leavers' slots (surplus arrivals appended, surplus holes filled from the tail) and returns the new row count. */
int plb_migrate_plan(plb_ctx* ctx, long long M, const double* d_tr_x, int nz, double Lz, int c0, int c1,
                     long long* h_counts);
int plb_migrate_apply(plb_ctx* ctx, long long M, int narr, double* const* h_arrs, const int* h_width,
                      long long capacity_rows, int nz, double Lz, int c0, int c1, long long* h_M_new);
int plb_halo_rows(plb_ctx* ctx, int narr, double* const* h_ptrs, const long long* h_row_doubles, int i0, int i1, int h);
/* Snapshot writer (pylamp_b200/output.py): move `count` doubles from rank `src` to rank 0 -- ncclSend on rank src,
 * ncclRecv into d_buf on rank 0, nothing on the other ranks or when src == 0 -- on the context's stream. */
int plb_comm_to_root(plb_ctx* ctx, int src, double* d_buf, long long count);
/* Snapshot reader: in-place ncclBroadcast of `count` doubles of d_buf from rank 0 to every rank on the context's
 * stream; nothing on one rank. */
int plb_comm_from_root(plb_ctx* ctx, double* d_buf, long long count);
void plb_comm_destroy(plb_ctx* ctx);

/* ---- snapshot output: pylamp2.py:637-650 writes tr_f as one row-major (M,13) array --------------------------
 * Rows [r0, r0+n) of ncol <= 16 fp64 columns (SoA; columns may alias each other) -> the row-major (n, ncol) block
 * d_out (which must not overlap a column).  n = 0 is a no-op.  Profiled as class 11, 16*ncol bytes per row. */
int plb_pack_columns(plb_ctx* ctx, long long r0, long long n, int ncol, const double* const* h_cols, double* d_out);
/* Snapshot reader, the reverse: of a chunk of n file rows -- d_x (n,2), d_f (n,ncol <= 16) and optionally d_v (n,2),
 * row-major, d_x 16-byte aligned -- the rows i in [r0, r1) whose cell row floor((nz-1)*z/Lz), clamped to [0, nz-2] (the migration's
 * rule), lies in [c0, c1) are appended in chunk order at row `base` of d_tr_x (rows of 2), the ncol columns h_cols
 * and, with d_v, d_trac_vel (rows of 2); base + selected rows must not exceed cap_rows.  d_tr_x == NULL: count only
 * (d_f may be NULL).  Synchronises once; *h_count = rows selected.  A row of the chunk with a non-finite z is an
 * error (nothing is written).  Profiled as class 11: 16 B per row counted, 8 * (2 + ncol + 2) B per row read and
 * per row written. */
int plb_unpack_rows(plb_ctx* ctx, long long n, const double* d_x, const double* d_f, int ncol, const double* d_v, int nz,
                    double Lz, int c0, int c1, long long r0, long long r1, long long base, long long cap_rows,
                    double* d_tr_x,
                    double* const* h_cols, double* d_trac_vel, long long* h_count);

/* ---- the marker->grid targets of one time step in ONE pass over the markers -------------------
 * (pylamp2.py:309-313 calls trac2grid four times -- nodes, cell centres, the two half-staggered grids --
 * and once more at :478; each call re-reads the coordinates and recomputes the cell of every marker.)
 * kind: 0 = (z-node, x-node), 1 = (z-mid, x-mid), 2 = (z-mid, x-node), 3 = (z-node, x-mid), where the
 * "mid" axes hold the midpoints of the node axis plus one point beyond the end (pylamp2.py:92-95).
 * axis_z/axis_x: the target's axes AFTER the ghost-node extension of pylamp_trac.py:207-217 (staggered
 * axes must carry >= 1 ghost node on the low side), crop_*: number of ghost nodes prepended.  Weighted
 * schemes only (PLB_AVG_ARITHMETIC|PLB_AVG_WEIGHTED, PLB_AVG_GEOMETRIC|PLB_AVG_WEIGHTED).  Every distinct
 * marker column is read once.  Returns 3, leaving the outputs untouched, when the request does not fit
 * (unweighted scheme, > 8 distinct columns, missing ghost node): use plb_trac2grid per target then. */
typedef struct {
    int kind;
    int k;
    const double* fields[PLB_MAX_FIELDS];
    int scheme[PLB_MAX_FIELDS];
    const double* axis_z;
    int nze;
    const double* axis_x;
    int nxe;
    int crop_z0, crop_x0;
    double* out[PLB_MAX_FIELDS];
} plb_t2g_target;
int plb_trac2grid_fused(plb_ctx* ctx, long long M, const double* d_tr_x, int nz, int nxx, int ld, double z0,
                        double zlen, double x0, double xlen, int ntargets, const plb_t2g_target* h_targets);

/* ---- marker-by-cell sort (device counting sort; no reference counterpart: NumPy's np.add.at at
 * pylamp_trac.py:257-298 is order-blind, on the GPU the order decides how well the node sums aggregate
 * and how local the gathers of grid2trac / RK are).  plb_sort_plan: d_dest[m] = slot of marker m in
 * cell-major order, cells numbered ie*(nxx-1)+je with the exact floor((n-1)*x/L) of pylamp2.py:588-589
 * (markers outside the box are clamped into the nearest cell); d_cell_start ((nz-1)*(nxx-1)+1 ints,
 * may be NULL) receives the first slot of every cell.  plb_permute: d_out[d_dest[m]] = d_in[m] for rows
 * of `width` (1 or 2) doubles; d_out must not alias d_in. */
int plb_sort_plan(plb_ctx* ctx, long long M, const double* d_tr_x, int nz, int nxx, double Lz, double Lx,
                  unsigned* d_dest, int* d_cell_start);
int plb_permute(plb_ctx* ctx, long long M, const unsigned* d_dest, const double* d_in, double* d_out, int width);

/* ---- markers -> grid: pylamp_trac.trac2grid, pylamp_trac.py:161-318 -------------------- */
/* h_out[4] = min z, max z, min x, max x over the markers (the ghost-node extension test of
 * pylamp_trac.py:207-217 is a global min/max).  Synchronises. */
int plb_marker_minmax(plb_ctx* ctx, long long M, const double* d_tr_x, double* h_out);
/* Average k marker columns to one target grid.  d_axis_z/d_axis_x are the (already ghost-
 * extended) target axes of length nze/nxe; the result is cropped to rows [crop_z0, crop_z0+nz)
 * and columns [crop_x0, crop_x0+nxx) and written to d_out[f] (nz x ld).  h_scheme[f] is the
 * reference's avgscheme bit-flag.  Empty nodes give 0/0 = NaN like the reference (:268).
 * z0/zlen/x0/xlen = axis[0] and axis[-1]-axis[0] as the host computed them (the cell lookup
 * floor((n-1)*(x-z0)/zlen) must round exactly like NumPy's, pylamp_trac.py:222-227). */
int plb_trac2grid(plb_ctx* ctx, long long M, const double* d_tr_x, int k,
                  const double* const* h_fields, const int* h_scheme,
                  const double* d_axis_z, int nze, const double* d_axis_x, int nxe,
                  double z0, double zlen, double x0, double xlen,
                  int crop_z0, int crop_x0, int nz, int nxx, int ld, double* const* h_out);

/* ---- grid -> markers: pylamp_trac.grid2trac, pylamp_trac.py:30-158 ---------------------- */
/* plb_trac2grid in two halves, for slab-owned markers (pylamp_b200/slabgrid.py; SURVEY.md 8e "halo-row
 * accumulate"): `scatter` zeroes d_planes and leaves the raw sums of this rank's markers in it --
 * planes [field 0..k-1 | sum of weights (if a weighted scheme is present) | marker count (if an
 * unweighted one is)], each nze*nxe over the extended axes, *h_nplanes of them -- without any
 * all-reduce; after the caller has combined the rows shared with the neighbouring slabs, `finalise`
 * divides / exponentiates rows [row0,row1) of the cropped (nz x nxx) target (pylamp_trac.py:276-316). */
int plb_trac2grid_scatter(plb_ctx* ctx, long long M, const double* d_tr_x, int k,
                          const double* const* h_fields, const int* h_scheme, const double* d_axis_z,
                          int nze, const double* d_axis_x, int nxe, double z0, double zlen, double x0,
                          double xlen, double* d_planes, int* h_nplanes);
int plb_trac2grid_finalise(plb_ctx* ctx, int k, const int* h_scheme, const double* d_planes, int nze, int nxe,
                           int crop_z0, int crop_x0, int nz, int nxx, int ld, int row0, int row1,
                           double* const* h_out);

/* method = PLB_METHOD_{NEAREST,LINEAR,VELDIV}.  Writes k output columns (SoA, length M).
 * Markers outside the grid get `defval` and are counted into *h_n_outside (synchronises). */
int plb_grid2trac(plb_ctx* ctx, long long M, const double* d_tr_x, int method, int k,
                  const double* const* h_fields, const double* d_grid_z, int nz,
                  const double* d_grid_x, int nxx, int ld, double z0, double zlen, double x0,
                  double xlen, double defval, double* const* h_out, long long* h_n_outside);

/* ---- marker advection: pylamp_trac.RK (order 4), pylamp_trac.py:321-388 ----------------- */
/* d_vz_c/d_vx_c: cell-centred velocities with BC ring, (nzc x ld) with nzc = nz+1, nxc = nxx+1;
 * d_gc_z/d_gc_x their coordinates.  x+ = x + (1/6) dt (k1+k2+k3+k4) (the reference's weights);
 * d_v_out = (x+ - x)/dt.  d_x_out, d_v_out are (M,2). */
int plb_rk4(plb_ctx* ctx, long long M, const double* d_tr_x, const double* d_vz_c,
            const double* d_vx_c, const double* d_gc_z, int nzc, const double* d_gc_x, int nxc,
            int ld, double z0, double zlen, double x0, double xlen, double dt, double* d_x_out,
            double* d_v_out);
/* plb_rk4 followed by plb_fence_count on the new positions in one pass over the markers (the positions are
 * final after the RK update: pylamp2.py:550, then the fence :558-572 and the per-cell count :588-593).
 * d_v_out holds (x_new - x_old)/dt of the UNfenced positions like the reference's trac_vel (pylamp_trac.py:386). */
int plb_rk4_fence_count(plb_ctx* ctx, long long M, const double* d_tr_x, const double* d_vz_c, const double* d_vx_c,
                        const double* d_gc_z, int nzc, const double* d_gc_x, int nxc, int ld, double z0, double zlen,
                        double x0, double xlen, double dt, double* d_x_out, double* d_v_out, double Lz, double Lx,
                        double eps, int nz, int nxx, long long* d_kelem, long long* d_count);

/* ---- driver-inline marker steps of pylamp2.py ------------------------------------------ */
/* fence, pylamp2.py:558-572 (fence enabled, no FLOWTHRU/CYCLIC): x<=0 -> eps, x>=L -> L-eps */
int plb_fence(plb_ctx* ctx, long long M, double* d_tr_x, double Lz, double Lx, double eps);
/* the same with a set of walls (bit 0 z = 0, bit 1 x = 0, bit 2 z = L, bit 3 x = L): markers beyond a wall whose bit is
 * clear -- a BC_TYPE_FLOWTHRU wall, pylamp2.py:565, :569 -- are left alone (the caller removes them, :573-581) */
int plb_fence_walls(plb_ctx* ctx, long long M, double* d_tr_x, double Lz, double Lx, double eps, int walls);
/* cell index + per-cell count, pylamp2.py:588-593.  BIT-EXACT parity item: ielem =
 * floor((nz-1)*z/Lz) with IEEE mul then div, kelem = ielem*(nxx-1)+jelem (int64);
 * d_count[(nz-1)*(nxx-1)] int64.  d_kelem may be NULL. */
int plb_cell_index_count(plb_ctx* ctx, long long M, const double* d_tr_x, int nz, int nxx,
                         double Lz, double Lx, long long* d_kelem, long long* d_count);
/* plb_fence followed by plb_cell_index_count in one pass over d_tr_x (pylamp2.py:558-572 then
 * :588-593; identical results, the coordinates are read once). */
int plb_fence_count(plb_ctx* ctx, long long M, double* d_tr_x, double Lz, double Lx, double eps, int nz,
                    int nxx, long long* d_kelem, long long* d_count);
/* marker property update, pylamp2.py:291-303 (columns of tr_f) */
int plb_update_properties(plb_ctx* ctx, long long M, int tdep_rho, int tdep_eta, double Tref,
                          double etamin, double etamax, double gasr, const double* d_T,
                          const double* d_rho0,
                          const double* d_alpha, const double* d_Ea, const double* d_eta0,
                          double* d_rho, double* d_eta);
/* cell-centre velocities + BC ghost ring, pylamp2.py:491-545; outputs (nz+1) x ldc */
int plb_centre_velocities(plb_ctx* ctx, int nz, int nxx, int ld, const double* d_vz,
                          const double* d_vx, const int* h_bc, int ldc, double* d_vz_c,
                          double* d_vx_c);
/* subgrid diffusion marker update, pylamp2.py:471-476:  Tsg = Told-(Told-T)*exp(-d*dt/tau),
 * d_dT = Tsg - T (stage 1);  T = Tsg - back (stage 2, after trac2grid/grid2trac of d_dT) */
int plb_subgrid_stage1(plb_ctx* ctx, long long M, double dt, double dz, double dx,
                       const double* d_Told, const double* d_T, const double* d_cp,
                       const double* d_rho, const double* d_k, double* d_Tsg, double* d_dT);
int plb_subgrid_stage2(plb_ctx* ctx, long long M, const double* d_Tsg, const double* d_back,
                       double* d_T);
/* fused form of the marker temperature update + subgrid diffusion, pylamp2.py:448-480 (same
 * arithmetic as grid2trac + the two stages above, one pass over the markers per stage):
 * stage 1: T1 = T + interp(d_field = T_new - T_grid); Tsg, dT from T (old) and T1; T is not written
 * stage 2: T = Tsg - interp(d_field = f_sgc).   Markers outside the grid are counted (stopOnError). */
int plb_subgrid_fused(plb_ctx* ctx, int stage, long long M, const double* d_tr_x, const double* d_field,
                      const double* d_grid_z, int nz, const double* d_grid_x, int nxx, int ld, double z0,
                      double zlen, double x0, double xlen, double dt, double dz, double dx, double* d_T,
                      const double* d_cp, const double* d_rho, const double* d_k, double* d_Tsg, double* d_dT,
                      long long* h_n_outside);
/* max over a field region / generic reductions used by the dt selection, pylamp2.py:339-366.
 * h_out = max of a (nz x nxx, ld) field (signed max, quirk 6).  Synchronises. */
int plb_field_max(plb_ctx* ctx, int nz, int nxx, int ld, const double* d_f, double* h_out);
/* max over nodes of 2*kz/(rho*cp): pylamp2.py:340-341.  Synchronises. */
int plb_max_diffusivity2(plb_ctx* ctx, int nz, int nxx, int ld, const double* d_kz,
                         const double* d_rho, const double* d_cp, double* h_out);

/* ---- Stokes operator: pylamp_stokes.makeStokesMatrix, pylamp_stokes.py:104-563 ----------- */
/* Matrix-free operator in the reference's exact DOF layout and row scaling, including ghost,
 * wall, corner and anchor rows.  h_grid_z/h_grid_x: node coordinates (any rectilinear spacing);
 * h_bc[4] indexed DIM*wall+dir = [z=0, x=0, z=L, x=L].  Supported: z-walls NOSLIP|FREESLIP,
 * x-walls FREESLIP (the reference itself is singular for NOSLIP x-walls, SURVEY.md quirk 4). */
int plb_stokes_create(plb_ctx* ctx, int nz, int nxx, int ld, const double* h_grid_z,
                      const double* h_grid_x, const int* h_bc, plb_stokes** out);
void plb_stokes_destroy(plb_stokes* op);
/* bind coefficient fields (nz x ld, device; must stay alive) and compute Kcont/Kbond
 * (pylamp_stokes.py:116-122) on the device.  gz, gx: gravity G (pylamp_const.py:21). */
int plb_stokes_set_coeffs(plb_stokes* op, const double* d_etas, const double* d_etan,
                          const double* d_rho, double gz, double gx);
/* h_out[2] = {Kcont, Kbond}.  Synchronises. */
int plb_stokes_scaling(plb_stokes* op, double* h_out);
/* rhs in the reference's interleaved layout, length 3*nz*nxx (pylamp_stokes.py:429, 490) */
int plb_stokes_rhs(plb_stokes* op, double* d_rhs);
/* y = A x, both interleaved [vz,vx,P] per node, length 3*nz*nxx (what A_ref @ x gives) */
int plb_stokes_apply(plb_stokes* op, const double* d_x, double* d_y);
/* replaces scipy.sparse.linalg.spsolve(csc_matrix(A), rhs) at pylamp2.py:360: solves A x = rhs
 * with flexible GCR + geometric multigrid.  d_rhs: interleaved right-hand side (NULL = the
 * system's own, as plb_stokes_rhs gives).  x interleaved like the reference's solution vector.
 * rtol is on the true residual in the viscosity-scaled norm (rows weighted by 1/sqrt|diag| resp.
 * sqrt(eta)/Kcont).  Returns non-zero (and still writes x) if not converged within maxit. */
int plb_stokes_solve(plb_stokes* op, const double* d_rhs, double rtol, int maxit, double* d_x,
                     int* h_iters, double* h_relres);
/* solver tuning: "nu" (Chebyshev steps per smoothing, default 3), "gcr_m" (truncation window, 30),
 * "coarsen_wide" (1: 4x4-cell viscosity averaging, stable with sharp contrasts; 0: 2x2),
 * "cheb_ratio" (8), "dense_max" (largest coarse level solved by a dense inverse, 640),
 * "nu_coarse" (60), "rtol_accept" (1e-8: a solve stalled at its fp64 floor is accepted below
 * this), "hydrostatic" (1: solve for the deviation from the lithostatic pressure), "warm_start"
 * (0: zero start, 1: start from the previous solve's iterate, 2: linear extrapolation of the last two), "reorth_thresh" (1e-4), "lmax_every" (1: the
 * smoother's eigenvalue estimates are recomputed on every n-th coefficient update) */
int plb_stokes_set_param(plb_stokes* op, const char* name, double value);
/* free-surface stabilisation terms of makeStokesMatrix(surfstab=True, tstep, surfstab_theta),
 * pylamp_stokes.py:422-426 and :483-487: theta_dt = surfstab_theta * tstep (<= 0: off).  Uses the
 * density field of the last plb_stokes_set_coeffs, which also switches the terms off again. */
int plb_stokes_set_surfstab(plb_stokes* op, double theta_dt);
/* test hook: one multigrid V-cycle x = V(b) on the velocity block; b, x are two planes
 * [vz | vx] of nz*nxx doubles each */
int plb_stokes_vcycle(plb_stokes* op, const double* d_b2, double* d_x2);
/* h_out[6] = {Krylov iterations, V-cycles, final scaled relative residual of the last solve,
 * fp64 residual floor met on the current coefficient fields (0 = none; reset by set_coeffs/set_surfstab),
 * status (0 converged to rtol; 1 stopped above rtol at the fp64 floor or at stagnation but accepted,
 * <= "rtol_accept"; 2 not converged), effective tolerance the solve iterated to} */
int plb_stokes_last_stats(plb_stokes* op, double* h_out);
/* x2vp, pylamp_stokes.py:86-101: de-interleave into three (nz x ld) planes */
int plb_x2vp(plb_ctx* ctx, int nz, int nxx, int ld, const double* d_x, double* d_vz,
             double* d_vx, double* d_p);

/* ---- energy operator: pylamp_diff.makeDiffusionMatrix, pylamp_diff.py:85-183 -------------- */
int plb_diff_create(plb_ctx* ctx, int nz, int nxx, int ld, const double* h_grid_z,
                    const double* h_grid_x, const double* h_gridmp_z, const double* h_gridmp_x,
                    const int* h_bc, const double* h_bcvalue, plb_diff** out);
void plb_diff_destroy(plb_diff* op);
int plb_diff_set_coeffs(plb_diff* op, const double* d_T, const double* d_kz, const double* d_kx,
                        const double* d_cp, const double* d_rho, const double* d_H, double tstep);
/* full-size (nz x ld) initial guess for the NEXT plb_diff_solve only (default: the field T); a time
 * loop passes T + (previous step's temperature increment) */
int plb_diff_set_initial_guess(plb_diff* op, const double* d_x0);
/* rhs / apply / solve on (nz x nxx) vectors stored with the leading dimension ld */
int plb_diff_rhs(plb_diff* op, double* d_rhs);
int plb_diff_apply(plb_diff* op, const double* d_x, double* d_y);
/* replaces spsolve at pylamp2.py:419: restarted GMRES on the row-scaled system, started from the
 * current temperature field.  d_rhs NULL = the system's own right-hand side. */
int plb_diff_solve(plb_diff* op, const double* d_rhs, double rtol, int maxit, double* d_x,
                   int* h_iters, double* h_relres);

#ifdef __cplusplus
}
#endif
#endif
