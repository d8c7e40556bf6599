// output.cu -- device side of the `.npz` snapshot writer (pylamp_b200/output.py; pylamp2.py:637-650).
//
// The reference writes its markers' properties as one row-major (M,13) array `tr_f`; here they live as 13
// separate columns (SoA).  plb_pack_columns turns a row range of the columns into that row-major block on the
// device, one chunk at a time, so that the host only ever receives bytes in file order.  A CTA stages a tile
// of PACK_ROWS rows x ncol columns in shared memory: it reads each column segment coalesced and writes the
// tile, which is one contiguous stretch of the output, coalesced.
//
// plb_unpack_rows is the reader's reverse (output.read_snapshot): a chunk of file rows -- tr_x (n,2), tr_f (n,ncol)
// and optionally tr_v (n,2), row-major as in the file -- is staged tile by tile in shared memory, the rows this rank
// owns are selected by their cell row (cell_row.cuh, the migration's rule) and appended, in file order, to the
// rank's tr_x, SoA columns and marker velocities.  Slots come from a count per tile and an exclusive scan over the
// tiles, so the order is deterministic.
#include "cell_row.cuh"
#include "common.cuh"

namespace {

constexpr int PACK_ROWS = 256;      // rows per tile = threads per CTA
constexpr int PACK_MAXCOL = 16;     // 256 x 16 x 8 B = 32 KB of shared memory

struct PackCols {
    const double* p[PACK_MAXCOL];
};

__global__ void __launch_bounds__(PACK_ROWS)
k_pack_columns(long long r0, long long n, int ncol, PackCols C, double* __restrict__ out) {
    __shared__ double tile[PACK_ROWS * PACK_MAXCOL];
    const long long ntiles = (n + PACK_ROWS - 1) / PACK_ROWS;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const long long row0 = t * PACK_ROWS;
        const int rows = (int)min((long long)PACK_ROWS, n - row0);
        if (threadIdx.x < rows) {
            const long long src = r0 + row0 + threadIdx.x;
#pragma unroll
            for (int c = 0; c < PACK_MAXCOL; c++)      // (static indices keep the pointers in the parameter bank)
                if (c < ncol) tile[threadIdx.x * ncol + c] = C.p[c][src];
        }
        __syncthreads();
        double* o = out + row0 * ncol;
        for (int i = threadIdx.x; i < rows * ncol; i += PACK_ROWS) o[i] = tile[i];
        __syncthreads();
    }
}

constexpr int UNPACK_ROWS = 256;    // rows per tile = threads per CTA (8 warps)

struct UnpackCols {
    double* p[PACK_MAXCOL];
};

// 1: selected (row i in the window [r0, r1) and its cell row in [c0, c1)), 0: not, -1: non-finite z (no owner)
__device__ __forceinline__ int unpack_class(long long i, double z, int nz, double Lz, int c0, int c1, long long r0,
                                            long long r1) {
    if (!isfinite(z)) return -1;
    const int r = row_of(z, nz, Lz);
    return i >= r0 && i < r1 && r >= c0 && r < c1 ? 1 : 0;
}

// pass 1: owned rows per tile; rows without an owner are counted in nbad
__global__ void __launch_bounds__(UNPACK_ROWS)
k_unpack_count(long long n, const double2* __restrict__ x, int nz, double Lz, int c0, int c1, long long r0,
               long long r1, long long* __restrict__ tile_cnt, unsigned long long* __restrict__ nbad) {
    __shared__ int wsum[UNPACK_ROWS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long ntiles = (n + UNPACK_ROWS - 1) / UNPACK_ROWS;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const long long i = t * UNPACK_ROWS + threadIdx.x;
        const int k = i < n ? unpack_class(i, x[i].x, nz, Lz, c0, c1, r0, r1) : 0;
        const unsigned sel = __ballot_sync(0xffffffffu, k == 1), bad = __ballot_sync(0xffffffffu, k < 0);
        if (lane == 0) {
            wsum[warp] = __popc(sel);
            if (bad) atomicAdd(nbad, (unsigned long long)__popc(bad));
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int s = 0;
            for (int w = 0; w < UNPACK_ROWS / 32; w++) s += wsum[w];
            tile_cnt[t] = s;
        }
        __syncthreads();
    }
}

// exclusive scan of the per-tile counts in place (one CTA of 1024 threads); *total = their sum
__global__ void __launch_bounds__(1024) k_unpack_scan(long long ntiles, long long* __restrict__ c, long long* __restrict__ total) {
    __shared__ long long wsum[32];
    __shared__ long long carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (long long b = 0; b < ntiles; b += 1024) {
        const long long i = b + threadIdx.x;
        const long long v = i < ntiles ? c[i] : 0;
        long long s = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        if (lane == 31) wsum[warp] = s;
        __syncthreads();
        if (warp == 0) {
            long long w = wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            wsum[lane] = w;
        }
        __syncthreads();
        const long long excl = carry + (warp ? wsum[warp - 1] : 0) + s - v;
        if (i < ntiles) c[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

// pass 2: stage the tile's rows (contiguous stretches of x, f and v: coalesced reads), compact the owned rows'
// tile positions with a block scan, write each output column / row pair as one contiguous stretch (coalesced)
__global__ void __launch_bounds__(UNPACK_ROWS)
k_unpack_scatter(long long n, const double* __restrict__ x, const double* __restrict__ f, int ncol,
                 const double* __restrict__ v, int nz, double Lz, int c0, int c1, long long r0, long long r1,
                 const long long* __restrict__ tile_off,
                 long long base, double* __restrict__ ox, UnpackCols D, double* __restrict__ ov) {
    __shared__ double tf[UNPACK_ROWS * PACK_MAXCOL];
    __shared__ double tx[UNPACK_ROWS * 2], tv[UNPACK_ROWS * 2];
    __shared__ int src[UNPACK_ROWS];
    __shared__ int wsum[UNPACK_ROWS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long ntiles = (n + UNPACK_ROWS - 1) / UNPACK_ROWS;
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const long long row0 = t * UNPACK_ROWS;
        const int rows = (int)min((long long)UNPACK_ROWS, n - row0);
        for (int i = threadIdx.x; i < rows * ncol; i += UNPACK_ROWS) tf[i] = f[row0 * ncol + i];
        for (int i = threadIdx.x; i < rows * 2; i += UNPACK_ROWS) {
            tx[i] = x[row0 * 2 + i];
            if (v) tv[i] = v[row0 * 2 + i];
        }
        __syncthreads();
        const bool sel = threadIdx.x < rows &&
                         unpack_class(row0 + threadIdx.x, tx[2 * threadIdx.x], nz, Lz, c0, c1, r0, r1) == 1;
        const unsigned b = __ballot_sync(0xffffffffu, sel);
        if (lane == 0) wsum[warp] = __popc(b);
        __syncthreads();
        int pre = __popc(b & ((1u << lane) - 1u)), cnt = 0;
        for (int w = 0; w < UNPACK_ROWS / 32; w++) {
            if (w < warp) pre += wsum[w];
            cnt += wsum[w];
        }
        if (sel) src[pre] = threadIdx.x;
        __syncthreads();
        const long long o = base + tile_off[t];
        if (threadIdx.x < cnt) {
            const int r = src[threadIdx.x];
#pragma unroll
            for (int c = 0; c < PACK_MAXCOL; c++)      // (static indices keep the pointers in the parameter bank)
                if (c < ncol) D.p[c][o + threadIdx.x] = tf[r * ncol + c];
        }
        for (int i = threadIdx.x; i < 2 * cnt; i += UNPACK_ROWS) {
            const int j = 2 * src[i >> 1] + (i & 1);
            ox[2 * o + i] = tx[j];
            if (ov) ov[2 * o + i] = tv[j];
        }
        __syncthreads();
    }
}

}  // namespace

extern "C" {

// Rows [r0, r0+n) of ncol fp64 columns (columns may alias each other) -> row-major (n, ncol) block at d_out,
// which must not overlap a column.  n = 0 is a no-op.
int plb_pack_columns(plb_ctx* ctx, long long r0, long long n, int ncol, const double* const* h_cols, double* d_out) {
    if (!ctx) return 1;
    if (r0 < 0 || n < 0) PLB_FAIL(ctx, "plb_pack_columns: bad row range r0=%lld n=%lld", r0, n);
    if (ncol < 1 || ncol > PACK_MAXCOL) PLB_FAIL(ctx, "plb_pack_columns: ncol=%d outside [1, %d]", ncol, PACK_MAXCOL);
    if (n == 0) return 0;
    if (!h_cols || !d_out) PLB_FAIL(ctx, "plb_pack_columns: null column array or output");
    PackCols C;
    for (int c = 0; c < ncol; c++) {
        if (!h_cols[c]) PLB_FAIL(ctx, "plb_pack_columns: column %d is null", c);
        C.p[c] = h_cols[c];
    }
    for (int c = ncol; c < PACK_MAXCOL; c++) C.p[c] = nullptr;
    PLB_CUDA(ctx, cudaSetDevice(ctx->device));
    plb_prof_scope prof_(ctx, PLB_K_MARKER_MISC, 16.0 * ncol * (double)n);
    k_pack_columns<<<plb_grid_for(ctx, n, PACK_ROWS, 8), PACK_ROWS, 0, ctx->stream>>>(r0, n, ncol, C, d_out);
    PLB_LAUNCHED(ctx);
    return 0;
}

// Appends the rows of a chunk of file rows that this rank keeps -- row i in [r0, r1) and cell row
// floor((nz-1)*z/Lz), clamped, in [c0, c1) -- in chunk order at row `base` of d_tr_x (rows of 2), the ncol SoA
// columns h_cols and, if d_v is given, d_trac_vel (rows of 2).  d_x (n,2), d_f (n,ncol), d_v (n,2): row-major.
// d_tr_x == NULL: count only (d_f may be NULL).  Synchronises once; *h_count = rows selected.  A row with a non-finite
// z, inside the window or not, has no owner: an error, and nothing is written.
int plb_unpack_rows(plb_ctx* ctx, long long n, const double* d_x, const double* d_f, int ncol, const double* d_v, int nz,
                    double Lz, int c0, int c1, long long r0, long long r1, long long base, long long cap_rows,
                    double* d_tr_x,
                    double* const* h_cols, double* d_trac_vel, long long* h_count) {
    if (!ctx) return 1;
    if (!h_count) PLB_FAIL(ctx, "plb_unpack_rows: null count");
    *h_count = 0;
    if (n < 0 || base < 0) PLB_FAIL(ctx, "plb_unpack_rows: bad rows n=%lld base=%lld", n, base);
    if (ncol < 1 || ncol > PACK_MAXCOL) PLB_FAIL(ctx, "plb_unpack_rows: ncol=%d outside [1, %d]", ncol, PACK_MAXCOL);
    if (nz < 2 || !(Lz > 0)) PLB_FAIL(ctx, "plb_unpack_rows: bad grid nz=%d Lz=%g", nz, Lz);
    if (n == 0) return 0;
    const bool fill = d_tr_x != nullptr;
    if (!d_x || (fill && !d_f)) PLB_FAIL(ctx, "plb_unpack_rows: null chunk");
    if ((uintptr_t)d_x % 16) PLB_FAIL(ctx, "plb_unpack_rows: the coordinates are not 16-byte aligned");
    UnpackCols D;
    for (int c = 0; c < PACK_MAXCOL; c++) D.p[c] = nullptr;
    if (fill) {
        if ((d_v == nullptr) != (d_trac_vel == nullptr))
            PLB_FAIL(ctx, "plb_unpack_rows: velocities need both the chunk's rows and the destination");
        if (!h_cols) PLB_FAIL(ctx, "plb_unpack_rows: null column array");
        for (int c = 0; c < ncol; c++) {
            if (!h_cols[c]) PLB_FAIL(ctx, "plb_unpack_rows: column %d is null", c);
            D.p[c] = h_cols[c];
        }
    }
    PLB_CUDA(ctx, cudaSetDevice(ctx->device));
    const long long ntiles = (n + UNPACK_ROWS - 1) / UNPACK_ROWS;
    if (plb_ws_reserve(ctx, (size_t)(ntiles + 2) * sizeof(long long))) return 2;
    long long* tile = (long long*)ctx->ws;
    long long* cnt = tile + ntiles;      // [0] rows selected, [1] rows with a non-finite z
    PLB_CUDA(ctx, cudaMemsetAsync(cnt, 0, 2 * sizeof(long long), ctx->stream));
    const int grid = plb_grid_for(ctx, n, UNPACK_ROWS, 8);
    {
        plb_prof_scope prof_(ctx, PLB_K_MARKER_MISC, 16.0 * (double)n);
        k_unpack_count<<<grid, UNPACK_ROWS, 0, ctx->stream>>>(n, (const double2*)d_x, nz, Lz, c0, c1, r0, r1, tile,
                                                              (unsigned long long*)(cnt + 1));
        PLB_LAUNCHED(ctx);
    }
    k_unpack_scan<<<1, 1024, 0, ctx->stream>>>(ntiles, tile, cnt);
    PLB_LAUNCHED(ctx);
    long long* h = (long long*)(ctx->h_pinned + 48);
    PLB_CUDA(ctx, cudaMemcpyAsync(h, cnt, 2 * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const long long total = h[0], bad = h[1];
    if (bad) PLB_FAIL(ctx, "plb_unpack_rows: %lld of %lld rows have a non-finite z (no owner)", bad, n);
    *h_count = total;
    if (!fill || total == 0) return 0;
    if (base + total > cap_rows)
        PLB_FAIL(ctx, "plb_unpack_rows: rows [%lld, %lld) exceed the %lld rows allocated", base, base + total, cap_rows);
    const double row_bytes = 8.0 * (2 + ncol + (d_v ? 2 : 0));
    plb_prof_scope prof_(ctx, PLB_K_MARKER_MISC, row_bytes * (double)(n + total));
    k_unpack_scatter<<<grid, UNPACK_ROWS, 0, ctx->stream>>>(n, d_x, d_f, ncol, d_v, nz, Lz, c0, c1, r0, r1, tile, base,
                                                           d_tr_x, D, d_trac_vel);
    PLB_LAUNCHED(ctx);
    return 0;
}

}  // extern "C"
