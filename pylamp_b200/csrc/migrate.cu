// migrate.cu -- marker migration between z-slabs (north_star: "markers migrate between owning slabs each step";
// replaces the reference's index-strided sharing + Allreduce of marker-sized arrays, pylamp2.py:445-455, :550-555).
//
// Rank r owns the markers whose cell row floor((nz-1)*z/Lz) (pylamp2.py:588) lies in [c0, c1).  After RK4 and
// the fence a marker has moved at most 0.45 cells, so leavers go to the slab directly below or above:
//   plan : one pass over the coordinates lists the leavers per direction (compaction by atomic slots), the two
//          counts are swapped with the neighbours (grouped ncclSend/ncclRecv) and read back together;
//   apply: the leavers' rows -- coordinates, every distinct property column, velocities -- are packed into one
//          payload per direction, exchanged with one grouped ncclSend/ncclRecv pair per neighbour, and the
//          arrivals are written into the leavers' slots; surplus arrivals are appended, surplus holes are filled
//          from the tail.  Only O(movers) entries of the marker arrays are touched.
// All marker kernels are order-independent, so which slot a marker lands in does not matter.
#include <vector>

#include "cell_row.cuh"
#include "comm.cuh"

struct plb_migrate_ws {
    int* idx[2] = {nullptr, nullptr};     // leavers going down / up
    long long cap_idx = 0;
    int* counts = nullptr;                // [0..1] leavers per direction, [2] too far, [3] low holes, [4] tail survivors
    double* xcnt = nullptr;               // 4 doubles: counts to / from the neighbours
    double *send = nullptr, *recv = nullptr;
    size_t cap_send = 0, cap_recv = 0;
    int *low = nullptr, *tail = nullptr;  // holes below the new end / survivors beyond it
    long long cap_low = 0;
    long long n_leave[2] = {0, 0}, n_arr[2] = {0, 0};
    long long M_plan = -1;
};

namespace {

__global__ void __launch_bounds__(256)
k_mig_list(long long M, const double2* __restrict__ trx, int nz, double Lz, int c0, int c1, int lo_ok, int hi_ok,
           int* __restrict__ idx_dn, int* __restrict__ idx_up, long long cap, int* __restrict__ counts) {
    for (long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
        const int ie = row_of(trx[m].x, nz, Lz);
        if (ie >= c0 && ie < c1) continue;
        const int dir = ie < c0 ? 0 : 1;
        if (ie < lo_ok || ie >= hi_ok) atomicAdd(counts + 2, 1);          // beyond the neighbouring slab
        const int slot = atomicAdd(counts + dir, 1);
        if (slot < cap) (dir ? idx_up : idx_dn)[slot] = (int)m;
    }
}

__global__ void k_mig_counts_to_double(const int* __restrict__ counts, double* __restrict__ x) {
    x[0] = counts[0], x[1] = counts[1], x[2] = 0, x[3] = 0;
}

struct MigArrays {
    double* p[20];
    int w[20];
    int off[20];       // column of the payload row
    int n, W;
};

__global__ void __launch_bounds__(256)
k_mig_pack(int n, const int* __restrict__ idx, MigArrays A, double* __restrict__ out) {
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
        const long long m = idx[t];
        double* row = out + (size_t)t * A.W;
        for (int a = 0; a < A.n; a++)
            for (int c = 0; c < A.w[a]; c++) row[A.off[a] + c] = A.p[a][m * A.w[a] + c];
    }
}

// holes below the new end of the arrays
__global__ void __launch_bounds__(256)
k_mig_low_holes(int n0, const int* __restrict__ i0, int n1, const int* __restrict__ i1, long long M_new,
                int* __restrict__ low, int* __restrict__ counts) {
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n0 + n1; t += gridDim.x * blockDim.x) {
        const int m = t < n0 ? i0[t] : i1[t - n0];
        if (m < M_new) low[atomicAdd(counts + 3, 1)] = m;
    }
}

// survivors in the tail [M_new, M): they move into the holes the arrivals did not fill
__global__ void __launch_bounds__(256)
k_mig_tail(long long M_new, long long M, const double2* __restrict__ trx, int nz, double Lz, int c0, int c1,
           int* __restrict__ tail, int* __restrict__ counts) {
    for (long long m = M_new + blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
        const int ie = row_of(trx[m].x, nz, Lz);
        if (ie >= c0 && ie < c1) tail[atomicAdd(counts + 4, 1)] = (int)m;
    }
}

// arrival t -> low[t] while holes last, then appended behind the old end
__global__ void __launch_bounds__(256)
k_mig_unpack(int n_arr, const double* __restrict__ in, const int* __restrict__ low, int n_low, long long M_old,
             MigArrays A) {
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n_arr; t += gridDim.x * blockDim.x) {
        const long long m = t < n_low ? (long long)low[t] : M_old + (t - n_low);
        const double* row = in + (size_t)t * A.W;
        for (int a = 0; a < A.n; a++)
            for (int c = 0; c < A.w[a]; c++) A.p[a][m * A.w[a] + c] = row[A.off[a] + c];
    }
}

__global__ void __launch_bounds__(256)
k_mig_fill(int n, const int* __restrict__ dst, const int* __restrict__ src, MigArrays A) {
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n; t += gridDim.x * blockDim.x) {
        const long long d = dst[t], s = src[t];
        for (int a = 0; a < A.n; a++)
            for (int c = 0; c < A.w[a]; c++) A.p[a][d * A.w[a] + c] = A.p[a][s * A.w[a] + c];
    }
}

// markers beyond the box (pylamp2.py:563-571: x <= 0 or x >= L in either direction)
__device__ __forceinline__ bool outside_box(const double2 p, double Lz, double Lx) {
    return p.x <= 0 || p.x >= Lz || p.y <= 0 || p.y >= Lx;
}

__global__ void __launch_bounds__(256)
k_del_list(long long M, const double2* __restrict__ trx, double Lz, double Lx, int* __restrict__ idx, long long cap,
           int* __restrict__ counts) {
    for (long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x)
        if (outside_box(trx[m], Lz, Lx)) {
            const int slot = atomicAdd(counts, 1);
            if (slot < cap) idx[slot] = (int)m;
        }
}

__global__ void __launch_bounds__(256)
k_del_tail(long long M_new, long long M, const double2* __restrict__ trx, double Lz, double Lx, int* __restrict__ tail,
           int* __restrict__ counts) {
    for (long long m = M_new + blockIdx.x * (long long)blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x)
        if (!outside_box(trx[m], Lz, Lx)) tail[atomicAdd(counts + 4, 1)] = (int)m;
}

template <typename T>
int grow(plb_ctx* ctx, T** p, size_t* cap, size_t need) {
    if (need <= *cap) return 0;
    PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (*p) cudaFree(*p);
    *p = nullptr, *cap = 0;
    const size_t want = need + need / 4 + 1024;
    PLB_CUDA(ctx, cudaMalloc(p, want * sizeof(T)));
    *cap = want;
    return 0;
}

}  // namespace

extern "C" {

// h_counts[4] = {leavers down, leavers up, arrivals from below, arrivals from above}.  Synchronises once.
int plb_migrate_plan(plb_ctx* ctx, long long M, const double* d_tr_x, int nz, double Lz, int c0, int c1,
                     long long* h_counts) {
    if (!ctx || !h_counts) return 1;
    if (M >= (1LL << 31)) PLB_FAIL(ctx, "plb_migrate_plan: %lld markers exceed the 32-bit index lists", M);
    PLB_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!ctx->mig) ctx->mig = new plb_migrate_ws();
    plb_migrate_ws* w = ctx->mig;
    if (!w->counts) {
        PLB_CUDA(ctx, cudaMalloc(&w->counts, 8 * sizeof(int)));
        PLB_CUDA(ctx, cudaMalloc(&w->xcnt, 8 * sizeof(double)));
    }
    const long long cap = M / 8 + 4096;            // a step moves far fewer markers across a slab boundary
    if (cap > w->cap_idx) {
        PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (int d = 0; d < 2; d++) {
            if (w->idx[d]) cudaFree(w->idx[d]);
            w->idx[d] = nullptr;
            PLB_CUDA(ctx, cudaMalloc(&w->idx[d], (size_t)cap * sizeof(int)));
        }
        w->cap_idx = cap;
    }
    const int R = plb_comm_size(ctx), rank = plb_comm_rank(ctx);
    PLB_CUDA(ctx, cudaMemsetAsync(w->counts, 0, 8 * sizeof(int), ctx->stream));
    // rows a leaver may be in: the neighbouring slabs (even split of the cell rows, like the slab solvers)
    const int rows = c1 - c0;
    const int lo_ok = rank > 0 ? c0 - rows : c0, hi_ok = rank < R - 1 ? c1 + rows + 1 : c1;
    if (M > 0) {
        k_mig_list<<<plb_grid_for(ctx, M, 256, 8), 256, 0, ctx->stream>>>(M, (const double2*)d_tr_x, nz, Lz, c0, c1, lo_ok, hi_ok,
                                                                        w->idx[0], w->idx[1], w->cap_idx, w->counts);
        PLB_LAUNCHED(ctx);
    }
    k_mig_counts_to_double<<<1, 1, 0, ctx->stream>>>(w->counts, w->xcnt);
    PLB_LAUNCHED(ctx);
    // my count going down is the lower neighbour's count of arrivals from above, and so on
    if (plb_comm_neighbour_exchange(ctx, w->xcnt + 0, 1, w->xcnt + 2, 1, w->xcnt + 1, 1, w->xcnt + 3, 1)) return 2;
    double h[4];
    int hc[4];
    PLB_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned, w->xcnt, 4 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    PLB_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + 8, w->counts, 4 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 4; i++) h[i] = ctx->h_pinned[i];
    memcpy(hc, ctx->h_pinned + 8, sizeof(hc));
    if (hc[2] > 0) PLB_FAIL(ctx, "plb_migrate_plan: %d markers moved beyond the neighbouring slab in one step", hc[2]);
    if (hc[0] > w->cap_idx || hc[1] > w->cap_idx)
        PLB_FAIL(ctx, "plb_migrate_plan: %d + %d leavers exceed the list capacity %lld", hc[0], hc[1], w->cap_idx);
    if ((rank == 0 && hc[0]) || (rank == R - 1 && hc[1]))
        PLB_FAIL(ctx, "plb_migrate_plan: markers outside the outer slabs (clamped rows cannot leave)");
    w->n_leave[0] = hc[0], w->n_leave[1] = hc[1];
    w->n_arr[0] = rank > 0 ? (long long)h[2] : 0, w->n_arr[1] = rank < R - 1 ? (long long)h[3] : 0;
    w->M_plan = M;
    h_counts[0] = w->n_leave[0], h_counts[1] = w->n_leave[1], h_counts[2] = w->n_arr[0], h_counts[3] = w->n_arr[1];
    return 0;
}

// Moves the rows planned by plb_migrate_plan.  h_arrs: narr arrays of `capacity_rows` rows of h_width[a] (1 or 2)
// doubles each, the first of which must be the coordinates; M rows are in use.  *h_M_new = rows in use afterwards.
int plb_migrate_apply(plb_ctx* ctx, long long M, int narr, double* const* h_arrs, const int* h_width,
                      long long capacity_rows, int nz, double Lz, int c0, int c1, long long* h_M_new) {
    if (!ctx || !ctx->mig || !h_M_new) return 1;
    plb_migrate_ws* w = ctx->mig;
    if (w->M_plan != M) PLB_FAIL(ctx, "plb_migrate_apply: no plan for %lld markers", M);
    if (narr < 1 || narr > 20 || h_width[0] != 2) PLB_FAIL(ctx, "plb_migrate_apply: 1..20 arrays, coordinates first");
    PLB_CUDA(ctx, cudaSetDevice(ctx->device));
    w->M_plan = -1;
    MigArrays A;
    A.n = narr, A.W = 0;
    for (int a = 0; a < narr; a++) {
        if (h_width[a] != 1 && h_width[a] != 2) PLB_FAIL(ctx, "plb_migrate_apply: width must be 1 or 2");
        A.p[a] = h_arrs[a], A.w[a] = h_width[a], A.off[a] = A.W, A.W += h_width[a];
    }
    const long long n_leave = w->n_leave[0] + w->n_leave[1], n_arr = w->n_arr[0] + w->n_arr[1];
    const long long M_new = M - n_leave + n_arr;
    if (M_new > capacity_rows || M + std::max(0LL, n_arr - n_leave) > capacity_rows)
        PLB_FAIL(ctx, "plb_migrate_apply: %lld rows needed, capacity %lld", M_new, capacity_rows);
    *h_M_new = M_new;
    if (n_leave == 0 && n_arr == 0) return 0;
    size_t cs = w->cap_send, cr = w->cap_recv;
    if (grow(ctx, &w->send, &cs, (size_t)n_leave * A.W + 2) || grow(ctx, &w->recv, &cr, (size_t)n_arr * A.W + 2)) return 2;
    w->cap_send = cs, w->cap_recv = cr;
    size_t cl = (size_t)w->cap_low;
    if ((size_t)n_leave + 2 > cl) {
        PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (w->low) cudaFree(w->low);
        if (w->tail) cudaFree(w->tail);
        w->low = w->tail = nullptr;
        const size_t want = (size_t)n_leave + n_leave / 4 + 1024;
        PLB_CUDA(ctx, cudaMalloc(&w->low, want * sizeof(int)));
        PLB_CUDA(ctx, cudaMalloc(&w->tail, want * sizeof(int)));
        w->cap_low = (long long)want;
    }
    // pack and exchange the payloads (down part first)
    double* send_up = w->send + (size_t)w->n_leave[0] * A.W;
    double* recv_up = w->recv + (size_t)w->n_arr[0] * A.W;
    for (int d = 0; d < 2; d++)
        if (w->n_leave[d]) {
            k_mig_pack<<<plb_grid_for(ctx, w->n_leave[d], 256, 4), 256, 0, ctx->stream>>>((int)w->n_leave[d], w->idx[d], A,
                                                                                       d ? send_up : w->send);
            PLB_LAUNCHED(ctx);
        }
    if (plb_comm_neighbour_exchange(ctx, w->send, (size_t)w->n_leave[0] * A.W, w->recv, (size_t)w->n_arr[0] * A.W, send_up,
                                    (size_t)w->n_leave[1] * A.W, recv_up, (size_t)w->n_arr[1] * A.W))
        return 2;
    // holes below the new end take the arrivals; what is left of them takes the survivors of the tail
    if (n_leave) {
        k_mig_low_holes<<<plb_grid_for(ctx, n_leave, 256, 4), 256, 0, ctx->stream>>>((int)w->n_leave[0], w->idx[0], (int)w->n_leave[1],
                                                                                  w->idx[1], M_new, w->low, w->counts);
        PLB_LAUNCHED(ctx);
    }
    if (M_new < M) {
        k_mig_tail<<<plb_grid_for(ctx, M - M_new, 256, 4), 256, 0, ctx->stream>>>(M_new, M, (const double2*)h_arrs[0], nz, Lz, c0, c1,
                                                                               w->tail, w->counts);
        PLB_LAUNCHED(ctx);
    }
    // number of low holes: all holes when the arrays do not shrink, else n_leave - (holes in the tail)
    int hc[2] = {0, 0};
    PLB_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + 16, w->counts + 3, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(hc, ctx->h_pinned + 16, sizeof(hc));
    const int n_low = hc[0], n_tail = hc[1];
    if (n_arr) {
        k_mig_unpack<<<plb_grid_for(ctx, n_arr, 256, 4), 256, 0, ctx->stream>>>((int)n_arr, w->recv, w->low, n_low, M, A);
        PLB_LAUNCHED(ctx);
    }
    if (n_low > n_arr) {
        if (n_tail != n_low - (int)n_arr)
            PLB_FAIL(ctx, "plb_migrate_apply: internal: %d tail survivors for %d open holes", n_tail, n_low - (int)n_arr);
        k_mig_fill<<<plb_grid_for(ctx, n_tail, 256, 4), 256, 0, ctx->stream>>>(n_tail, w->low + n_arr, w->tail, A);
        PLB_LAUNCHED(ctx);
    }
    return 0;
}

// Removes the markers beyond the box from all arrays (pylamp2.py:563-581: with the fence disabled, or beyond a
// flow-through wall, the reference flags them TR__ID = -1 and np.delete's their rows): the survivors of the tail move
// into the holes (marker order is free), *h_M_new rows remain.  Coordinates first in h_arrs.  Synchronises twice.
int plb_delete_outside(plb_ctx* ctx, long long M, int narr, double* const* h_arrs, const int* h_width, double Lz, double Lx,
                       long long* h_M_new) {
    if (!ctx || !h_M_new) return 1;
    if (M >= (1LL << 31)) PLB_FAIL(ctx, "plb_delete_outside: too many markers for the 32-bit index lists");
    if (narr < 1 || narr > 20 || h_width[0] != 2) PLB_FAIL(ctx, "plb_delete_outside: 1..20 arrays, coordinates first");
    PLB_CUDA(ctx, cudaSetDevice(ctx->device));
    *h_M_new = M;
    if (M <= 0) return 0;
    if (!ctx->mig) ctx->mig = new plb_migrate_ws();
    plb_migrate_ws* w = ctx->mig;
    if (!w->counts) {
        PLB_CUDA(ctx, cudaMalloc(&w->counts, 8 * sizeof(int)));
        PLB_CUDA(ctx, cudaMalloc(&w->xcnt, 8 * sizeof(double)));
    }
    const long long cap = M / 8 + 4096;
    if (cap > w->cap_idx) {
        PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (int d = 0; d < 2; d++) {
            if (w->idx[d]) cudaFree(w->idx[d]);
            w->idx[d] = nullptr;
            PLB_CUDA(ctx, cudaMalloc(&w->idx[d], (size_t)cap * sizeof(int)));
        }
        w->cap_idx = cap;
    }
    MigArrays A;
    A.n = narr, A.W = 0;
    for (int a = 0; a < narr; a++) {
        if (h_width[a] != 1 && h_width[a] != 2) PLB_FAIL(ctx, "plb_delete_outside: width must be 1 or 2");
        A.p[a] = h_arrs[a], A.w[a] = h_width[a], A.off[a] = A.W, A.W += h_width[a];
    }
    const double2* x = (const double2*)h_arrs[0];
    PLB_CUDA(ctx, cudaMemsetAsync(w->counts, 0, 8 * sizeof(int), ctx->stream));
    k_del_list<<<plb_grid_for(ctx, M, 256, 8), 256, 0, ctx->stream>>>(M, x, Lz, Lx, w->idx[0], w->cap_idx, w->counts);
    PLB_LAUNCHED(ctx);
    int hc[5];
    PLB_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + 32, w->counts, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(hc, ctx->h_pinned + 32, sizeof(int));
    const long long n_del = hc[0];
    if (n_del == 0) return 0;
    if (n_del > w->cap_idx) {
        // more than an eighth of the cloud is outside: list them all (rare: a second pass with a full-size list)
        PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (int d = 0; d < 2; d++) {
            cudaFree(w->idx[d]);
            w->idx[d] = nullptr;
            PLB_CUDA(ctx, cudaMalloc(&w->idx[d], (size_t)(n_del + 1024) * sizeof(int)));
        }
        w->cap_idx = n_del + 1024;
        PLB_CUDA(ctx, cudaMemsetAsync(w->counts, 0, 8 * sizeof(int), ctx->stream));
        k_del_list<<<plb_grid_for(ctx, M, 256, 8), 256, 0, ctx->stream>>>(M, x, Lz, Lx, w->idx[0], w->cap_idx, w->counts);
        PLB_LAUNCHED(ctx);
    }
    const long long M_new = M - n_del;
    if ((long long)n_del + 2 > w->cap_low) {
        PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (w->low) cudaFree(w->low);
        if (w->tail) cudaFree(w->tail);
        w->low = w->tail = nullptr;
        const size_t want = (size_t)n_del + n_del / 4 + 1024;
        PLB_CUDA(ctx, cudaMalloc(&w->low, want * sizeof(int)));
        PLB_CUDA(ctx, cudaMalloc(&w->tail, want * sizeof(int)));
        w->cap_low = (long long)want;
    }
    k_mig_low_holes<<<plb_grid_for(ctx, n_del, 256, 4), 256, 0, ctx->stream>>>((int)n_del, w->idx[0], 0, w->idx[1], M_new, w->low,
                                                                            w->counts);
    PLB_LAUNCHED(ctx);
    k_del_tail<<<plb_grid_for(ctx, M - M_new, 256, 4), 256, 0, ctx->stream>>>(M_new, M, x, Lz, Lx, w->tail, w->counts);
    PLB_LAUNCHED(ctx);
    PLB_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned + 32, w->counts + 3, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PLB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(hc, ctx->h_pinned + 32, 2 * sizeof(int));
    if (hc[0] != hc[1]) PLB_FAIL(ctx, "plb_delete_outside: internal: %d holes below the new end, %d survivors beyond it", hc[0], hc[1]);
    if (hc[0] > 0) {
        k_mig_fill<<<plb_grid_for(ctx, hc[0], 256, 4), 256, 0, ctx->stream>>>(hc[0], w->low, w->tail, A);
        PLB_LAUNCHED(ctx);
    }
    *h_M_new = M_new;
    return 0;
}

void plb_migrate_free(plb_ctx* ctx) {
    if (!ctx || !ctx->mig) return;
    plb_migrate_ws* w = ctx->mig;
    void* ptrs[] = {w->idx[0], w->idx[1], w->counts, w->xcnt, w->send, w->recv, w->low, w->tail};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    delete w;
    ctx->mig = nullptr;
}

}  // extern "C"
