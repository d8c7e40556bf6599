// comm.cu -- one NCCL communicator per context (one process per GPU) for the z-slab solver:
// halo rows over NVLink with grouped ncclSend/ncclRecv, Krylov dot products and the other small
// reductions with ncclAllReduce.  NCCL is loaded with dlopen at run time (torch has normally loaded
// its bundled libnccl.so.2 already, which is then reused), so the library has no link-time
// dependency on it and single-GPU use never touches it.
#include <dlfcn.h>

#include <algorithm>

#include "comm.cuh"

namespace {

// the few NCCL entry points used (signatures from nccl.h 2.27/2.28; ABI-stable since 2.7)
typedef struct { char internal[128]; } nccl_uid;
typedef void* nccl_comm_t;
enum { NCCL_SUM = 0, NCCL_MAX = 2, NCCL_MIN = 3, NCCL_DOUBLE = 8 };

struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(nccl_uid*) = nullptr;
    int (*CommInitRank)(nccl_comm_t*, int, nccl_uid, int) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*Send)(const void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*Recv)(void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*Broadcast)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
} api;

int load_api(plb_ctx* ctx) {
    if (api.lib) return 0;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (api.lib) break;
    }
    if (!api.lib) PLB_FAIL(ctx, "plb_comm: cannot dlopen libnccl.so.2 (%s)", dlerror());
#define SYM(field, name)                                                     \
    *(void**)(&api.field) = dlsym(api.lib, name);                            \
    if (!api.field) PLB_FAIL(ctx, "plb_comm: NCCL symbol %s not found", name)
    SYM(GetUniqueId, "ncclGetUniqueId");
    SYM(CommInitRank, "ncclCommInitRank");
    SYM(CommDestroy, "ncclCommDestroy");
    SYM(AllReduce, "ncclAllReduce");
    SYM(Send, "ncclSend");
    SYM(Recv, "ncclRecv");
    SYM(Broadcast, "ncclBroadcast");
    SYM(GroupStart, "ncclGroupStart");
    SYM(GroupEnd, "ncclGroupEnd");
    SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
    return 0;
}

#define PLB_NCCL(ctx, call)                                                                     \
    do {                                                                                        \
        int r_ = (call);                                                                        \
        if (r_ != 0) PLB_FAIL(ctx, "%s:%d: %s: %s", __FILE__, __LINE__, #call, api.GetErrorString(r_)); \
    } while (0)

}  // namespace

struct plb_comm {
    int rank = 0, size = 1;
    nccl_comm_t comm = nullptr;
};

int plb_comm_rank(const plb_ctx* ctx) { return ctx->comm ? ctx->comm->rank : 0; }
int plb_comm_size(const plb_ctx* ctx) { return ctx->comm ? ctx->comm->size : 1; }

int plb_comm_allreduce(plb_ctx* ctx, double* d_buf, size_t count, int op) {
    if (!ctx->comm || ctx->comm->size == 1) return 0;
    int nop = op == PLB_OP_SUM ? NCCL_SUM : (op == PLB_OP_MAX ? NCCL_MAX : NCCL_MIN);
    PLB_NCCL(ctx, api.AllReduce(d_buf, d_buf, count, NCCL_DOUBLE, nop, ctx->comm->comm, ctx->stream));
    return 0;
}

// Exchange one halo row per plane with the z-neighbours.  `base` points at local row 0 of plane 0;
// local rows are [lo, hi] in global numbering with owned rows [r0, r1): rank > 0 has a halo row
// below (lo = r0 - 1), rank < size-1 one above (hi = r1).
int plb_comm_halo_exchange(plb_ctx* ctx, double* base, int nplanes, size_t plane_stride, int ld, int ncols,
                           int lo, int r0, int r1) {
    plb_comm* c = ctx->comm;
    if (!c || c->size == 1) return 0;
    const bool has_dn = c->rank > 0, has_up = c->rank < c->size - 1;
    PLB_NCCL(ctx, api.GroupStart());
    for (int p = 0; p < nplanes; p++) {
        double* pl = base + (size_t)p * plane_stride;
        if (has_dn) {
            // my first owned row -> lower neighbour's upper halo; its last owned row -> my lower halo
            PLB_NCCL(ctx, api.Send(pl + (size_t)(r0 - lo) * ld, ncols, NCCL_DOUBLE, c->rank - 1, c->comm, ctx->stream));
            PLB_NCCL(ctx, api.Recv(pl + (size_t)(r0 - 1 - lo) * ld, ncols, NCCL_DOUBLE, c->rank - 1, c->comm, ctx->stream));
        }
        if (has_up) {
            PLB_NCCL(ctx, api.Send(pl + (size_t)(r1 - 1 - lo) * ld, ncols, NCCL_DOUBLE, c->rank + 1, c->comm, ctx->stream));
            PLB_NCCL(ctx, api.Recv(pl + (size_t)(r1 - lo) * ld, ncols, NCCL_DOUBLE, c->rank + 1, c->comm, ctx->stream));
        }
    }
    PLB_NCCL(ctx, api.GroupEnd());
    return 0;
}

int plb_comm_halo_rows(plb_ctx* ctx, int narr, double* const* arrs, const long long* row_doubles, int i0, int i1, int h) {
    plb_comm* c = ctx->comm;
    if (!c || c->size == 1 || h <= 0) return 0;
    const bool has_dn = c->rank > 0, has_up = c->rank < c->size - 1;
    PLB_NCCL(ctx, api.GroupStart());
    for (int a = 0; a < narr; a++) {
        const size_t rd = (size_t)row_doubles[a];
        double* p = arrs[a];
        if (has_dn) {
            PLB_NCCL(ctx, api.Send(p + (size_t)i0 * rd, h * rd, NCCL_DOUBLE, c->rank - 1, c->comm, ctx->stream));
            PLB_NCCL(ctx, api.Recv(p + (size_t)(i0 - h) * rd, h * rd, NCCL_DOUBLE, c->rank - 1, c->comm, ctx->stream));
        }
        if (has_up) {
            PLB_NCCL(ctx, api.Send(p + (size_t)(i1 - h) * rd, h * rd, NCCL_DOUBLE, c->rank + 1, c->comm, ctx->stream));
            PLB_NCCL(ctx, api.Recv(p + (size_t)i1 * rd, h * rd, NCCL_DOUBLE, c->rank + 1, c->comm, ctx->stream));
        }
    }
    PLB_NCCL(ctx, api.GroupEnd());
    return 0;
}

int plb_comm_neighbour_exchange(plb_ctx* ctx, const double* send_dn, size_t n_send_dn, double* recv_dn, size_t n_recv_dn,
                                const double* send_up, size_t n_send_up, double* recv_up, size_t n_recv_up) {
    plb_comm* c = ctx->comm;
    if (!c || c->size == 1) return 0;
    const bool has_dn = c->rank > 0, has_up = c->rank < c->size - 1;
    PLB_NCCL(ctx, api.GroupStart());
    if (has_dn && n_send_dn) PLB_NCCL(ctx, api.Send(send_dn, n_send_dn, NCCL_DOUBLE, c->rank - 1, c->comm, ctx->stream));
    if (has_dn && n_recv_dn) PLB_NCCL(ctx, api.Recv(recv_dn, n_recv_dn, NCCL_DOUBLE, c->rank - 1, c->comm, ctx->stream));
    if (has_up && n_send_up) PLB_NCCL(ctx, api.Send(send_up, n_send_up, NCCL_DOUBLE, c->rank + 1, c->comm, ctx->stream));
    if (has_up && n_recv_up) PLB_NCCL(ctx, api.Recv(recv_up, n_recv_up, NCCL_DOUBLE, c->rank + 1, c->comm, ctx->stream));
    PLB_NCCL(ctx, api.GroupEnd());
    return 0;
}

namespace {
__global__ void __launch_bounds__(256) k_add_rows(long long n, const double* __restrict__ src, double* __restrict__ dst) {
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x)
        dst[t] += src[t];
}
}  // namespace

int plb_comm_accumulate_rows(plb_ctx* ctx, int narr, double* const* arrs, const long long* row_doubles,
                             const int* i0, const int* i1, const int* nrows, int h, double* scratch) {
    plb_comm* c = ctx->comm;
    if (!c || c->size == 1 || h <= 0) return 0;
    const bool has_dn = c->rank > 0, has_up = c->rank < c->size - 1;
    // what the neighbours wrote into my first / last h rows arrives in scratch, then is added
    PLB_NCCL(ctx, api.GroupStart());
    size_t off = 0;
    for (int a = 0; a < narr; a++) {
        const size_t rd = (size_t)row_doubles[a];
        double* p = arrs[a];
        if ((has_dn && i0[a] < h) || (has_up && nrows[a] - i1[a] < h) || i1[a] - i0[a] < h)
            PLB_FAIL(ctx, "plb_comm_accumulate_rows: slab [%d, %d) of %d rows is too thin for %d boundary rows", i0[a], i1[a], nrows[a], h);
        const int hd = h, hu = h;
        if (has_dn) {
            PLB_NCCL(ctx, api.Send(p + (size_t)(i0[a] - hd) * rd, hd * rd, NCCL_DOUBLE, c->rank - 1, c->comm, ctx->stream));
            PLB_NCCL(ctx, api.Recv(scratch + off, h * rd, NCCL_DOUBLE, c->rank - 1, c->comm, ctx->stream));
        }
        off += h * rd;
        if (has_up) {
            PLB_NCCL(ctx, api.Send(p + (size_t)i1[a] * rd, hu * rd, NCCL_DOUBLE, c->rank + 1, c->comm, ctx->stream));
            PLB_NCCL(ctx, api.Recv(scratch + off, h * rd, NCCL_DOUBLE, c->rank + 1, c->comm, ctx->stream));
        }
        off += h * rd;
    }
    PLB_NCCL(ctx, api.GroupEnd());
    off = 0;
    for (int a = 0; a < narr; a++) {
        const size_t rd = (size_t)row_doubles[a];
        double* p = arrs[a];
        const long long n = (long long)h * rd;
        // the lower neighbour's rows [its i1, its i1 + h) are my rows [i0, i0 + h); the upper one's
        // [its i0 - h, its i0) are my [i1 - h, i1)
        if (has_dn) {
            k_add_rows<<<plb_grid_for(ctx, n, 256, 4), 256, 0, ctx->stream>>>(n, scratch + off, p + (size_t)i0[a] * rd);
            PLB_LAUNCHED(ctx);
        }
        off += h * rd;
        if (has_up) {
            k_add_rows<<<plb_grid_for(ctx, n, 256, 4), 256, 0, ctx->stream>>>(n, scratch + off, p + (size_t)(i1[a] - h) * rd);
            PLB_LAUNCHED(ctx);
        }
        off += h * rd;
    }
    return 0;
}

extern "C" {

int plb_ctx_set_slab(plb_ctx* ctx, int i0, int i1, int halo) {
    if (!ctx) return 1;
    if (i1 < i0 || halo < 0) PLB_FAIL(ctx, "plb_ctx_set_slab: bad row range [%d, %d) / halo %d", i0, i1, halo);
    ctx->slab_i0 = i0, ctx->slab_i1 = i1, ctx->slab_halo = halo;
    ctx->slab_on = i1 > i0;
    return 0;
}

int plb_halo_rows(plb_ctx* ctx, int narr, double* const* h_ptrs, const long long* h_row_doubles, int i0, int i1, int h) {
    if (!ctx) return 1;
    PLB_CUDA(ctx, cudaSetDevice(ctx->device));
    return plb_comm_halo_rows(ctx, narr, h_ptrs, h_row_doubles, i0, i1, h);
}

int plb_comm_unique_id(plb_ctx* ctx, char* h_id128) {
    if (!ctx || !h_id128) return 1;
    if (load_api(ctx)) return 2;
    nccl_uid id;
    PLB_NCCL(ctx, api.GetUniqueId(&id));
    memcpy(h_id128, id.internal, 128);
    return 0;
}

int plb_comm_init(plb_ctx* ctx, int rank, int size, const char* h_id128) {
    if (!ctx || size < 1 || rank < 0 || rank >= size) return 1;
    if (ctx->comm) PLB_FAIL(ctx, "plb_comm_init: communicator already initialised");
    if (load_api(ctx)) return 2;
    PLB_CUDA(ctx, cudaSetDevice(ctx->device));
    plb_comm* c = new plb_comm();
    c->rank = rank, c->size = size;
    nccl_uid id;
    memcpy(id.internal, h_id128, 128);
    int r = api.CommInitRank(&c->comm, size, id, rank);
    if (r != 0) {
        delete c;
        PLB_FAIL(ctx, "ncclCommInitRank: %s", api.GetErrorString(r));
    }
    ctx->comm = c;
    return 0;
}

int plb_comm_info(plb_ctx* ctx, int* h_rank, int* h_size) {
    if (!ctx) return 1;
    *h_rank = plb_comm_rank(ctx), *h_size = plb_comm_size(ctx);
    return 0;
}

// in-place all-reduce of a device buffer of doubles (op: 0 sum, 1 max, 2 min) on the context's stream
int plb_allreduce(plb_ctx* ctx, double* d_buf, long long count, int op) {
    if (!ctx) return 1;
    PLB_CUDA(ctx, cudaSetDevice(ctx->device));
    return plb_comm_allreduce(ctx, d_buf, (size_t)count, op);
}

// point-to-point move of `count` doubles from rank `src` to rank 0 on the context's stream (snapshot writer):
// rank src sends d_buf, rank 0 receives into d_buf, every other rank (and src == 0) does nothing
int plb_comm_to_root(plb_ctx* ctx, int src, double* d_buf, long long count) {
    if (!ctx) return 1;
    plb_comm* c = ctx->comm;
    const int size = c ? c->size : 1;
    if (src < 0 || src >= size || count < 0) PLB_FAIL(ctx, "plb_comm_to_root: src %d of %d ranks, count %lld", src, size, count);
    if (size == 1 || src == 0 || count == 0 || (c->rank != src && c->rank != 0)) return 0;
    if (!d_buf) PLB_FAIL(ctx, "plb_comm_to_root: null buffer");
    PLB_CUDA(ctx, cudaSetDevice(ctx->device));
    if (c->rank == src)
        PLB_NCCL(ctx, api.Send(d_buf, (size_t)count, NCCL_DOUBLE, 0, c->comm, ctx->stream));
    else
        PLB_NCCL(ctx, api.Recv(d_buf, (size_t)count, NCCL_DOUBLE, src, c->comm, ctx->stream));
    return 0;
}

// in-place broadcast of `count` doubles from rank 0 to every rank on the context's stream (snapshot reader);
// nothing on one rank
int plb_comm_from_root(plb_ctx* ctx, double* d_buf, long long count) {
    if (!ctx) return 1;
    plb_comm* c = ctx->comm;
    if (count < 0) PLB_FAIL(ctx, "plb_comm_from_root: count %lld", count);
    if (!c || c->size == 1 || count == 0) return 0;
    if (!d_buf) PLB_FAIL(ctx, "plb_comm_from_root: null buffer");
    PLB_CUDA(ctx, cudaSetDevice(ctx->device));
    PLB_NCCL(ctx, api.Broadcast(d_buf, d_buf, (size_t)count, NCCL_DOUBLE, 0, c->comm, ctx->stream));
    return 0;
}

void plb_comm_destroy(plb_ctx* ctx) {
    if (!ctx || !ctx->comm) return;
    if (ctx->comm->comm) api.CommDestroy(ctx->comm->comm);
    delete ctx->comm;
    ctx->comm = nullptr;
}

}  // extern "C"
