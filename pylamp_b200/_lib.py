"""ctypes binding of libpylamp_b200.so (the C-ABI of include/pylamp_b200.h).

The product path has no CPU fallback: if the shared library is missing, or no CUDA device is
visible when a context is requested, this module raises.
"""
import ctypes as C
import os
import threading

from . import build as _build

_c_double_p = C.POINTER(C.c_double)
VP = C.c_void_p          # device pointers travel as integers (tensor.data_ptr())
LL = C.c_longlong
I = C.c_int
D = C.c_double
PP = C.POINTER(C.c_void_p)   # host array of device pointers
IP = C.POINTER(C.c_int)
DP = C.POINTER(C.c_double)   # host doubles

_PROTOS = {
    "plb_version": (C.c_char_p, []),
    "plb_ctx_create": (I, [I, C.POINTER(VP)]),
    "plb_ctx_destroy": (None, [VP]),
    "plb_ctx_set_stream": (I, [VP, VP]),
    "plb_ctx_sync": (I, [VP]),
    "plb_last_error": (C.c_char_p, [VP]),
    "plb_launch_count": (LL, [VP]),
    "plb_ctx_set_param": (I, [VP, C.c_char_p, D]),
    "plb_profile_enable": (I, [VP, I]),
    "plb_profile_read": (I, [VP, C.POINTER(LL), DP, DP]),
    "plb_comm_unique_id": (I, [VP, C.c_char_p]),
    "plb_comm_init": (I, [VP, I, I, C.c_char_p]),
    "plb_comm_info": (I, [VP, IP, IP]),
    "plb_allreduce": (I, [VP, VP, LL, I]),
    "plb_comm_destroy": (None, [VP]),
    "plb_comm_to_root": (I, [VP, I, VP, LL]),
    "plb_pack_columns": (I, [VP, LL, LL, I, PP, VP]),
    "plb_comm_from_root": (I, [VP, VP, LL]),
    "plb_unpack_rows": (I, [VP, LL, VP, VP, I, VP, I, D, I, I, LL, LL, LL, LL, VP, PP, VP, C.POINTER(LL)]),
    "plb_ctx_set_slab": (I, [VP, I, I, I]),
    "plb_inject_plan": (I, [VP, LL, VP, I, I, LL, LL, C.POINTER(LL)]),
    "plb_inject_apply": (I, [VP, LL, VP, VP, VP, I, PP, I, D, VP, VP, I, C.c_ulonglong, C.c_ulonglong]),
    "plb_delete_outside": (I, [VP, LL, I, PP, IP, D, D, C.POINTER(LL)]),
    "plb_migrate_plan": (I, [VP, LL, VP, I, D, I, I, C.POINTER(LL)]),
    "plb_migrate_apply": (I, [VP, LL, I, PP, IP, LL, I, D, I, I, C.POINTER(LL)]),
    "plb_halo_rows": (I, [VP, I, PP, C.POINTER(LL), I, I, I]),
    "plb_marker_minmax": (I, [VP, LL, VP, DP]),
    "plb_sort_plan": (I, [VP, LL, VP, I, I, D, D, VP, VP]),
    "plb_permute": (I, [VP, LL, VP, VP, VP, I]),
    "plb_trac2grid": (I, [VP, LL, VP, I, PP, IP, VP, I, VP, I, D, D, D, D, I, I, I, I, I, PP]),
    "plb_trac2grid_scatter": (I, [VP, LL, VP, I, PP, IP, VP, I, VP, I, D, D, D, D, VP, IP]),
    "plb_trac2grid_finalise": (I, [VP, I, IP, VP, I, I, I, I, I, I, I, I, I, PP]),
    "plb_grid2trac": (I, [VP, LL, VP, I, I, PP, VP, I, VP, I, I, D, D, D, D, D, PP,
                          C.POINTER(LL)]),
    "plb_rk4": (I, [VP, LL, VP, VP, VP, VP, I, VP, I, I, D, D, D, D, D, VP, VP]),
    "plb_rk4_fence_count": (I, [VP, LL, VP, VP, VP, VP, I, VP, I, I, D, D, D, D, D, VP, VP, D, D, D, I, I, VP, VP]),
    "plb_fence": (I, [VP, LL, VP, D, D, D]),
    "plb_fence_walls": (I, [VP, LL, VP, D, D, D, I]),
    "plb_cell_index_count": (I, [VP, LL, VP, I, I, D, D, VP, VP]),
    "plb_fence_count": (I, [VP, LL, VP, D, D, D, I, I, VP, VP]),
    "plb_update_properties": (I, [VP, LL, I, I, D, D, D, D, VP, VP, VP, VP, VP, VP, VP]),
    "plb_centre_velocities": (I, [VP, I, I, I, VP, VP, IP, I, VP, VP]),
    "plb_subgrid_stage1": (I, [VP, LL, D, D, D, VP, VP, VP, VP, VP, VP, VP]),
    "plb_subgrid_stage2": (I, [VP, LL, VP, VP, VP]),
    "plb_subgrid_fused": (I, [VP, I, LL, VP, VP, VP, I, VP, I, I, D, D, D, D, D, D, D, VP, VP, VP, VP, VP, VP,
                              C.POINTER(LL)]),
    "plb_field_max": (I, [VP, I, I, I, VP, DP]),
    "plb_max_diffusivity2": (I, [VP, I, I, I, VP, VP, VP, DP]),
    "plb_stokes_create": (I, [VP, I, I, I, DP, DP, IP, C.POINTER(VP)]),
    "plb_stokes_destroy": (None, [VP]),
    "plb_stokes_set_coeffs": (I, [VP, VP, VP, VP, D, D]),
    "plb_stokes_scaling": (I, [VP, DP]),
    "plb_stokes_rhs": (I, [VP, VP]),
    "plb_stokes_apply": (I, [VP, VP, VP]),
    "plb_stokes_solve": (I, [VP, VP, D, I, VP, IP, DP]),
    "plb_stokes_set_param": (I, [VP, C.c_char_p, D]),
    "plb_stokes_set_surfstab": (I, [VP, D]),
    "plb_stokes_vcycle": (I, [VP, VP, VP]),
    "plb_stokes_last_stats": (I, [VP, DP]),
    "plb_x2vp": (I, [VP, I, I, I, VP, VP, VP, VP]),
    "plb_diff_create": (I, [VP, I, I, I, DP, DP, DP, DP, IP, DP, C.POINTER(VP)]),
    "plb_diff_destroy": (None, [VP]),
    "plb_diff_set_coeffs": (I, [VP, VP, VP, VP, VP, VP, VP, D]),
    "plb_diff_set_initial_guess": (I, [VP, VP]),
    "plb_diff_rhs": (I, [VP, VP]),
    "plb_diff_apply": (I, [VP, VP, VP]),
    "plb_diff_solve": (I, [VP, VP, D, I, VP, IP, DP]),
}



class T2GTarget(C.Structure):
    """plb_t2g_target of include/pylamp_b200.h"""
    _fields_ = [("kind", C.c_int), ("k", C.c_int), ("fields", C.c_void_p * 8), ("scheme", C.c_int * 8),
                ("axis_z", C.c_void_p), ("nze", C.c_int), ("axis_x", C.c_void_p), ("nxe", C.c_int),
                ("crop_z0", C.c_int), ("crop_x0", C.c_int), ("out", C.c_void_p * 8)]


_PROTOS["plb_trac2grid_fused"] = (I, [VP, LL, VP, I, I, I, D, D, D, D, I, C.POINTER(T2GTarget)])

_lib = None
_lock = threading.Lock()


class PlbError(RuntimeError):
    pass


def load():
    """Load the shared library (raises if it has not been built)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = _build.lib_path()
        if not os.path.exists(path):
            raise PlbError(
                "libpylamp_b200.so not found at %s -- run `python -m pylamp_b200.build` "
                "(there is no CPU fallback)" % path)
        lib = C.CDLL(path)
        for name, (res, args) in _PROTOS.items():
            try:
                fn = getattr(lib, name)
            except AttributeError:
                continue          # reported by exported_symbols()/tests, raised on first use
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def exported(name):
    try:
        getattr(load(), name)
        return True
    except AttributeError:
        return False


class Context:
    """One plb_ctx per GPU: stream, scratch and error text."""

    def __init__(self, device=0):
        import torch
        if not torch.cuda.is_available():
            raise PlbError("pylamp_b200 needs a CUDA device (no CPU fallback)")
        self.lib = load()
        self.device = int(device)
        h = VP()
        rc = self.lib.plb_ctx_create(self.device, C.byref(h))
        if rc != 0:
            raise PlbError("plb_ctx_create(device=%d) failed with %d" % (device, rc))
        self.h = h
        self.slab = None
        # run on torch's current stream so that torch allocations/copies order with our kernels
        self.torch_device = torch.device("cuda", self.device)
        stream = torch.cuda.current_stream(self.torch_device)
        self.check(self.lib.plb_ctx_set_stream(self.h, VP(stream.cuda_stream)))

    def check(self, rc):
        if rc != 0:
            raise PlbError(self.lib.plb_last_error(self.h).decode() or "error %d" % rc)

    def call(self, name, *args):
        self.check(getattr(self.lib, name)(self.h, *args))

    def sync(self):
        self.check(self.lib.plb_ctx_sync(self.h))

    def init_comm(self, group=None):
        """Create this context's NCCL communicator for the z-slab solver: rank 0 makes the unique id,
        torch.distributed (any backend) broadcasts it, every rank joins.  One process per GPU."""
        import torch
        import torch.distributed as dist
        rank, size = dist.get_rank(group), dist.get_world_size(group)
        if size == 1:
            return 0, 1
        buf = C.create_string_buffer(128)
        if rank == 0:
            self.call("plb_comm_unique_id", buf)
        dev = self.torch_device if dist.get_backend(group) == "nccl" else torch.device("cpu")
        t = torch.frombuffer(bytearray(buf.raw), dtype=torch.uint8).clone().to(dev)
        dist.broadcast(t, src=0, group=group)
        ident = bytes(t.cpu().numpy().tobytes())
        self.call("plb_comm_init", rank, size, C.create_string_buffer(ident, 128))
        self.rank, self.size = rank, size
        return rank, size

    def set_slab(self, i0, i1, halo=3):
        """Slab-local grid fields (plb_ctx_set_slab): this rank keeps node rows [i0, i1) of every field current,
        plus `halo` rows of each z-neighbour; i1 <= i0 switches back to replicated fields."""
        self.call("plb_ctx_set_slab", int(i0), int(i1), int(halo))
        self.slab = (int(i0), int(i1), int(halo)) if i1 > i0 else None

    def halo_rows(self, tensors, h=None):
        """Exchange halo rows of full-size (nz, ...) float64 tensors with both z-neighbours (plb_halo_rows)."""
        i0, i1, halo = self.slab
        arr = ptr_array(tensors)
        rd = (LL * len(tensors))(*[int(t[0].numel()) for t in tensors])
        self.call("plb_halo_rows", len(tensors), arr, rd, i0, i1, halo if h is None else int(h))

    def comm_info(self):
        r, s = C.c_int(0), C.c_int(1)
        self.call("plb_comm_info", C.byref(r), C.byref(s))
        return r.value, s.value

    def allreduce(self, tensor, op="sum"):
        """In-place all-reduce of a float64 CUDA tensor over the slab communicator (no-op for 1 rank)."""
        self.call("plb_allreduce", tensor.data_ptr(), tensor.numel(), {"sum": 0, "max": 1, "min": 2}[op])
        return tensor

    def set_param(self, name, value):
        """Tuning knob of the context (include/pylamp_b200.h: plb_ctx_set_param)."""
        self.call("plb_ctx_set_param", name.encode(), float(value))

    def profile(self, on=True):
        self.call("plb_profile_enable", 1 if on else 0)

    def profile_read(self):
        """{class index: (launch count, total ms, algorithmic bytes)} since the last read."""
        cnt, ms, by = (LL * 16)(), (D * 16)(), (D * 16)()
        self.call("plb_profile_read", cnt, ms, by)
        return {i: (int(cnt[i]), float(ms[i]), float(by[i])) for i in range(16) if cnt[i]}

    @property
    def launches(self):
        return int(self.lib.plb_launch_count(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.plb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = {}


def default_context(device=None):
    import torch
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    ctx = _default_ctx.get(device)
    if ctx is None:
        ctx = _default_ctx[device] = Context(device)
    return ctx


def ptr_array(tensors):
    """Host array of device pointers from a list of tensors (kept alive by the caller)."""
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


def int_array(vals):
    return (C.c_int * len(vals))(*[int(v) for v in vals])


def dbl_array(vals):
    return (C.c_double * len(vals))(*[float(v) for v in vals])
