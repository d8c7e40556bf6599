// output.cu -- device side of the `.npz` snapshot writer (pylamp_b200/output.py; pylamp2.py:637-650).
//
// The reference writes its markers' properties as one row-major (M,13) array `tr_f`; here they live as 13
// separate columns (SoA).  plb_pack_columns turns a row range of the columns into that row-major block on the
// device, one chunk at a time, so that the host only ever receives bytes in file order.  A CTA stages a tile
// of PACK_ROWS rows x ncol columns in shared memory: it reads each column segment coalesced and writes the
// tile, which is one contiguous stretch of the output, coalesced.
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

}  // extern "C"
