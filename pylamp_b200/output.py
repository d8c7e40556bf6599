"""The reference's per-step `.npz` snapshots (pylamp2.py:637-650) on any number of ranks.

`write_snapshot(s, prefix, it)` writes `griddata.<it>.npz` (gridz, gridx, velz, velx, pres, rho, temp, tstep,
time) and `tracs.<it>.npz` (tr_x (M,2), tr_f (M,13), tr_v (M,2)) with the keys, dtypes and shapes the reference
writes, so that its pylamp_post.py reads them unchanged.  It is collective over the ranks of the context's
communicator; only rank 0 writes files.

The grids are five (nz, nxx) planes: rank 0 assembles them (`driver.full_field` when the fields are slab-local)
and writes them with np.savez.  The markers are streamed, so that host memory stays bounded at any marker count:
per array, per rank, per chunk of at most CHUNK_BYTES, the owning rank produces the chunk on the device (tr_f:
`plb_pack_columns` turns the 13 SoA columns into the reference's row-major rows; tr_x / tr_v: the contiguous row
slice as it is), `plb_comm_to_root` moves it to rank 0 if another rank owns it, and rank 0 copies it into one of
two pinned host buffers on a side stream while it writes the previous chunk into the zip member (CRC32 + file
write).  Rows are in rank order, and within a rank in the order of its arrays.  See DESIGN.md section 8.

`read_snapshot(prefix, it, o)` reads such a pair back into a `driver.State` that `driver.timestep` continues, on
any number of ranks, whatever number of ranks wrote it.  Rank 0 reads the grid file with np.load and the marker
members front to back through zipfile (CRC32 checked) in chunks of rows, in a worker thread one chunk ahead, into
one of two pinned host buffers; each chunk goes to the device, to every rank (`plb_comm_from_root`), and
`plb_unpack_rows` appends the rows the rank keeps (its slab's markers with `o.marker_ownership="slab"`, an even
split of the file's rows with "index") to its marker arrays.
"""
import ctypes as C
import os
import time
import zipfile
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

from . import _lib
from .pylamp_const import IX, IZ

# bytes per chunk: two device and two pinned host buffers of this size per rank
CHUNK_BYTES = 256 << 20

TRACS_MEMBERS = (("tr_x", 2), ("tr_f", 13), ("tr_v", 2))


def pack_columns(ctx, cols, r0, n, out=None):
    """Rows [r0, r0+n) of the float64 device columns `cols` (SoA; they may alias each other) as the row-major
    (n, len(cols)) block of the reference's tr_f layout (plb_pack_columns).  `out`: n*len(cols) doubles."""
    k = len(cols)
    if out is None:
        out = torch.empty((n, k), dtype=torch.float64, device=ctx.torch_device)
    for c in cols:
        if c.dtype != torch.float64 or not c.is_contiguous() or c.shape[0] < r0 + n:
            raise ValueError("pack_columns: columns must be contiguous float64 with at least %d rows" % (r0 + n))
    if out.numel() < n * k or out.dtype != torch.float64 or not out.is_contiguous():
        raise ValueError("pack_columns: out needs %d contiguous float64 elements" % (n * k))
    ctx.call("plb_pack_columns", int(r0), int(n), k, _lib.ptr_array(cols), out.data_ptr())
    return out


def plan_chunks(counts, widths):
    """(member, rank, first row, rows) of every chunk in file order: per member (array of `widths[m]` float64
    columns), per rank (`counts[m][r]` rows), per chunk of at most CHUNK_BYTES.  Every rank walks this same list."""
    jobs = []
    for m, w in enumerate(widths):
        step = max(1, CHUNK_BYTES // (8 * w))
        for r, n in enumerate(counts[m]):
            for a in range(0, n, step):
                jobs.append((m, r, a, min(step, n - a)))
    return jobs


def write_npz_stream(path, members, chunks):
    """Write float64 arrays to an uncompressed `.npz` that np.load reads like np.savez output (one ZIP64 member
    `<name>.npy` per array, format 1.0 header) without holding any array in memory.  members: [(name, shape)] in
    file order; chunks: iterable of (member index, bytes-like) in file order whose bytes, per member, concatenate
    to the array's C-order bytes.  Returns the seconds spent in the members' writes (CRC32 + file write)."""
    write_s = 0.0
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_STORED, allowZip64=True) as zf:
        state = {"m": -1, "f": None, "left": 0}

        def advance(to):            # close the open member, open (and for empty ones close) members up to `to`
            while state["m"] < to:
                if state["f"] is not None:
                    if state["left"]:
                        raise ValueError("write_npz_stream: member %s is %d bytes short"
                                         % (members[state["m"]][0], state["left"]))
                    state["f"].close()
                    state["f"] = None
                state["m"] += 1
                if state["m"] < len(members):
                    name, shape = members[state["m"]]
                    state["f"] = zf.open(name + ".npy", "w", force_zip64=True)
                    np.lib.format.write_array_header_1_0(
                        state["f"], {"descr": np.lib.format.dtype_to_descr(np.dtype(np.float64)),
                                     "fortran_order": False, "shape": tuple(int(d) for d in shape)})
                    state["left"] = 8 * int(np.prod(shape))

        for m, buf in chunks:
            if m != state["m"]:
                if m < state["m"]:
                    raise ValueError("write_npz_stream: chunks out of member order")
                advance(m)
            nbytes = memoryview(buf).nbytes
            if nbytes > state["left"]:
                raise ValueError("write_npz_stream: member %s overflows" % members[m][0])
            t0 = time.perf_counter()
            state["f"].write(buf)
            write_s += time.perf_counter() - t0
            state["left"] -= nbytes
        advance(len(members))
    return write_s


def _device_chunks(s, jobs, widths, stats):
    """The chunks of `jobs` as they reach rank 0's pinned buffers: yields (member, uint8 ndarray) on rank 0 (after
    enqueuing the next chunk's pack / receive / copy), nothing on the other ranks (which pack and send theirs)."""
    ctx = s.ctx
    rank, _ = ctx.comm_info()
    dev = ctx.torch_device
    main = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(dev)
    x, v = s.tr_x.contiguous(), s.trac_vel.contiguous()
    cols = [c if c.is_contiguous() else c.contiguous() for c in s.cols]
    # device buffers: packed tr_f chunks of this rank, and on rank 0 the chunks received from the others
    need_dev = any((m == 1 and r == rank) or (rank == 0 and r != 0) for m, r, _, _ in jobs)
    dbuf = [torch.empty(CHUNK_BYTES // 8, dtype=torch.float64, device=dev) for _ in range(2)] if need_dev else None
    hbuf = [torch.empty(CHUNK_BYTES, dtype=torch.uint8, pin_memory=True) for _ in range(2)] \
        if rank == 0 and jobs else None
    done = [None, None]          # rank 0: the D2H copy out of dbuf[i] / into hbuf[i] has finished
    timed = []
    prev = None
    for k, (m, r, a, n) in enumerate(jobs):
        if rank != r and rank != 0:
            continue
        i, w = k % 2, widths[m]
        cnt = n * w
        if done[i] is not None:
            main.wait_event(done[i])         # dbuf[i] is free again
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record(main)
        if rank == r:
            if m == 1:
                chunk = pack_columns(ctx, cols, a, n, dbuf[i][:cnt])
            else:
                chunk = (x if m == 0 else v).view(-1)[a * w:(a + n) * w]
            if r != 0:
                ctx.call("plb_comm_to_root", r, chunk.data_ptr(), cnt)
                continue
        else:
            chunk = dbuf[i][:cnt]
            ctx.call("plb_comm_to_root", r, chunk.data_ptr(), cnt)
        # rank 0: device chunk -> pinned hbuf[i] on the side stream (hbuf[i] was written out two chunks ago)
        ready = torch.cuda.Event()
        ready.record(main)
        side.wait_event(ready)
        with torch.cuda.stream(side):
            hbuf[i][:8 * cnt].view(torch.float64).copy_(chunk, non_blocking=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record(side)
        done[i] = e1
        timed.append((e0, e1))
        if prev is not None:
            yield _landed(prev, stats)
        prev = (m, e1, hbuf[i].numpy()[:8 * cnt])
    if prev is not None:
        yield _landed(prev, stats)
    torch.cuda.synchronize(dev)
    stats["device_ms"] = sum(e0.elapsed_time(e1) for e0, e1 in timed)
    stats["chunks"] = len(timed)


def _landed(prev, stats):
    m, ev, view = prev
    t0 = time.perf_counter()
    ev.synchronize()
    stats["wait_s"] += time.perf_counter() - t0
    return m, view


def write_snapshot(s, prefix, it=None):
    """Write `<prefix>griddata.<it>.npz` and `<prefix>tracs.<it>.npz` (it: s.it by default) from the state `s` of
    every rank.  Collective and synchronous: call it on every rank; it returns once rank 0 has closed both files.
    Returns rank 0's timings {"griddata_s", "write_s" (tracs CRC32 + file write), "wait_s" (host waiting for
    chunks), "device_ms" (sum over the chunks of pack + NCCL + D2H, CUDA events), "chunks", "bytes"}."""
    from .driver import full_field
    it = s.it if it is None else it
    if s.newvel is None or s.trac_vel is None:
        raise TypeError("write_snapshot: no time step has run yet (no velocity fields / marker velocities)")
    ctx = s.ctx
    rank, world = ctx.comm_info()
    dev = ctx.torch_device
    stats = {"griddata_s": 0.0, "write_s": 0.0, "wait_s": 0.0, "device_ms": 0.0, "chunks": 0, "bytes": 0}
    # grids: full_field all-reduces the owners' rows of slab-local fields (a no-op on replicated ones)
    planes = {"velz": s.newvel[IZ], "velx": s.newvel[IX], "pres": s.newpres, "rho": s.f_rho, "temp": s.newtemp}
    planes = {k: (np.zeros(tuple(s.nx)) if f is None else full_field(s, f)) for k, f in planes.items()}
    gpath, tpath = "%sgriddata.%d.npz" % (prefix, it), "%stracs.%d.npz" % (prefix, it)
    if rank == 0:
        t0 = time.perf_counter()
        host = {k: (f.detach().cpu().numpy() if isinstance(f, torch.Tensor) else f) for k, f in planes.items()}
        np.savez(gpath, gridz=s.grid[IZ], gridx=s.grid[IX], velz=host["velz"], velx=host["velx"], pres=host["pres"],
                 rho=host["rho"], temp=host["temp"], tstep=it, time=s.totaltime)
        stats["griddata_s"] = time.perf_counter() - t0
    # markers: rows of every array on every rank, then the chunks in file order.  (trac_vel keeps the rows of the
    # last advection: the injection of pylamp2.py:594-633 appends to tr_x and tr_f only.)
    M = s.tr_x.shape[0]
    if any(c.shape[0] < M for c in s.cols):
        raise ValueError("write_snapshot: tr_x has %d rows, the columns %s"
                         % (M, sorted({c.shape[0] for c in s.cols})))
    cnt = torch.zeros((len(TRACS_MEMBERS), world), dtype=torch.float64, device=dev)
    cnt[:, rank] = torch.tensor([M, M, s.trac_vel.shape[0]], dtype=torch.float64)
    counts = [[int(c) for c in row] for row in ctx.allreduce(cnt.view(-1)).view(cnt.shape).tolist()]
    widths = [w for _, w in TRACS_MEMBERS]
    jobs = plan_chunks(counts, widths)
    chunks = _device_chunks(s, jobs, widths, stats)
    if rank == 0:
        members = [(name, (sum(counts[m]), w)) for m, (name, w) in enumerate(TRACS_MEMBERS)]
        stats["write_s"] = write_npz_stream(tpath, members, chunks)
        stats["bytes"] = os.path.getsize(gpath) + os.path.getsize(tpath)
    else:
        for _ in chunks:
            pass
    # every rank returns after rank 0 has closed the files
    ctx.allreduce(torch.zeros(1, dtype=torch.float64, device=dev))
    torch.cuda.synchronize(dev)
    return stats


# --------------------------------------------------------------------------------------------------------------------
# reader

READ_PIECE = 16 << 20       # bytes per zipfile read: the transient host copy besides the two pinned chunk buffers
GRID_KEYS = ("gridz", "gridx", "velz", "velx", "pres", "rho", "temp", "tstep", "time")
_ZIP_ERRORS = (zipfile.BadZipFile, EOFError, OSError, zlib.error, ValueError)


def read_plan(M):
    """(first row, rows) of the chunks the reader walks in file order: at most CHUNK_BYTES of tr_f per chunk; the
    tr_x and tr_v chunks cover the same rows."""
    step = max(1, CHUNK_BYTES // (8 * TRACS_MEMBERS[1][1]))
    return [(a, min(step, M - a)) for a in range(0, M, step)]


def index_split(M, world):
    """Row bounds of marker_ownership="index": rank r keeps the file rows [b[r], b[r+1]) = [r*M//W, (r+1)*M//W).
    (The file does not record which rank wrote which rows, so this is an even split, not the writer's split.)"""
    return [(r * int(M)) // int(world) for r in range(int(world) + 1)]


def _bad(path, member, what):
    return ValueError("%s: member %s: %s" % (path, member, what))


class _Member:
    """A float64 (rows, width) `.npy` member of an `.npz`, read front to back through zipfile's reader, which checks
    the member's CRC32 when its end is reached; stored and deflated members alike."""

    def __init__(self, zf, path, name, width):
        self.path, self.name, self.width = path, name, width
        try:
            self.f = zf.open(name + ".npy")
            version = np.lib.format.read_magic(self.f)
            if version == (1, 0):
                shape, fortran, dtype = np.lib.format.read_array_header_1_0(self.f)
            elif version == (2, 0):
                shape, fortran, dtype = np.lib.format.read_array_header_2_0(self.f)
            else:
                raise ValueError("unsupported .npy format version %d.%d" % version)
        except _ZIP_ERRORS as e:
            raise _bad(path, name, e) from e
        if dtype != np.dtype("<f8"):
            raise _bad(path, name, "dtype %s, expected little-endian float64 ('<f8')" % dtype.str)
        if fortran:
            raise _bad(path, name, "Fortran order, expected C order")
        if len(shape) != 2 or shape[1] != width:
            raise _bad(path, name, "shape %s, expected (rows, %d)" % (shape, width))
        self.rows = int(shape[0])

    def read_into(self, out):
        """Fill the uint8 array `out` with the member's next len(out) bytes."""
        pos, n = 0, out.shape[0]
        while pos < n:
            try:
                b = self.f.read(min(READ_PIECE, n - pos))
            except _ZIP_ERRORS as e:
                raise _bad(self.path, self.name, e) from e
            if not b:
                raise _bad(self.path, self.name, "%d bytes short of its %d rows" % (n - pos, self.rows))
            out[pos:pos + len(b)] = np.frombuffer(b, dtype=np.uint8)
            pos += len(b)

    def finish(self):
        """The member must end here (reading up to its end also completes the CRC32 check)."""
        try:
            extra = self.f.read(1)
        except _ZIP_ERRORS as e:
            raise _bad(self.path, self.name, e) from e
        if extra:
            raise _bad(self.path, self.name, "longer than its %d rows" % self.rows)

    def close(self):
        self.f.close()


class TracsReader:
    """A `tracs.<it>.npz` opened for streaming: tr_x (M,2), tr_f (M,13), tr_v (Mv,2) validated from their `.npy`
    headers (`M`, `Mv`); `open(names)` gives members positioned at their first row, for `read_rows`."""

    def __init__(self, path):
        self.path = path
        try:
            self.zf = zipfile.ZipFile(path)
        except (zipfile.BadZipFile, EOFError, ValueError) as e:
            raise ValueError("%s: not a readable .npz: %s" % (path, e)) from e
        try:
            names = set(self.zf.namelist())
            rows = {}
            for name, w in TRACS_MEMBERS:
                if name + ".npy" not in names:
                    raise _bad(path, name, "missing")
                m = _Member(self.zf, path, name, w)
                rows[name] = m.rows
                m.close()
            if rows["tr_f"] != rows["tr_x"]:
                raise _bad(path, "tr_f", "%d rows, tr_x has %d" % (rows["tr_f"], rows["tr_x"]))
        except BaseException:
            self.zf.close()
            raise
        self.M, self.Mv = rows["tr_x"], rows["tr_v"]

    def open(self, names):
        return [_Member(self.zf, self.path, name, dict(TRACS_MEMBERS)[name]) for name in names]

    def close(self):
        self.zf.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def read_rows(members, n, out):
    """The next n rows of each member in turn into the float64 array `out`, back to back (n*width doubles each).
    Returns the number of doubles written."""
    off = 0
    for m in members:
        k = n * m.width
        m.read_into(out[off:off + k].view(np.uint8))
        off += k
    return off


def read_griddata(path):
    """The arrays of a `griddata.<it>.npz`, checked: every key of the reference's file; gridz / gridx exactly
    `make_grids(nx, L)` with nx = their lengths and L = their last values; the planes (nz, nxx) float64; tstep an
    integer and time a number.  Returns {key: array}, with "nx" and "L" added."""
    from .setups import make_grids
    try:
        with np.load(path, allow_pickle=False) as g:
            for k in GRID_KEYS:
                if k not in g.files:
                    raise _bad(path, k, "missing")
            d = {}
            for k in GRID_KEYS:
                try:
                    d[k] = g[k]
                except _ZIP_ERRORS as e:
                    raise _bad(path, k, e) from e
    except (zipfile.BadZipFile, EOFError) as e:
        raise ValueError("%s: not a readable .npz: %s" % (path, e)) from e
    for k in ("gridz", "gridx"):
        a = d[k]
        if a.dtype != np.float64 or a.ndim != 1 or a.shape[0] < 2:
            raise _bad(path, k, "dtype %s, shape %s: expected a float64 axis of at least 2 nodes" % (a.dtype, a.shape))
    nx = (d["gridz"].shape[0], d["gridx"].shape[0])
    L = (float(d["gridz"][-1]), float(d["gridx"][-1]))
    grid, _ = make_grids(nx, L)
    for k, i in (("gridz", IZ), ("gridx", IX)):
        if not np.array_equal(d[k], grid[i]):
            raise _bad(path, k, "not the grid make_grids(%s, %s) builds" % (list(nx), list(L)))
    for k in ("velz", "velx", "pres", "rho", "temp"):
        if d[k].shape != nx or d[k].dtype != np.float64:
            raise _bad(path, k, "dtype %s, shape %s: expected float64 %s" % (d[k].dtype, d[k].shape, nx))
    if d["tstep"].shape != () or d["tstep"].dtype.kind not in "iu":
        raise _bad(path, "tstep", "expected an integer, got %s %s" % (d["tstep"].dtype, d["tstep"].shape))
    if d["time"].shape != () or d["time"].dtype.kind not in "iuf":
        raise _bad(path, "time", "expected a number, got %s %s" % (d["time"].dtype, d["time"].shape))
    d["nx"], d["L"] = nx, L
    return d


def _chunks_to_device(ctx, reader, path, names, plan, stats):
    """Every rank: yields (first row, rows, {member: (rows, width) device view}) per chunk of `plan` once the chunk's
    rows of the members `names` are in this rank's device buffer.  Rank 0 reads chunk k+1 from the file in a worker
    thread into one of two pinned buffers while chunk k goes to the device (copy_, plb_comm_from_root) and is
    consumed.  The double behind a chunk's rows carries rank 0's status, so that every rank stops at a chunk rank 0
    could not read."""
    rank, world = ctx.comm_info()
    dev = ctx.torch_device
    widths = dict(TRACS_MEMBERS)
    per_row = sum(widths[k] for k in names)
    nmax = max((n for _, n in plan), default=0)
    if not plan:
        return
    dbuf = torch.empty(per_row * nmax + 1, dtype=torch.float64, device=dev)
    stats["device_buffer_bytes"] = max(stats.get("device_buffer_bytes", 0), dbuf.numel() * 8)
    pool, members, fut = None, [], None
    if rank == 0:
        hbuf = [torch.empty(per_row * nmax + 1, dtype=torch.float64, pin_memory=True) for _ in range(2)]
        stats["pinned_bytes"] = max(stats.get("pinned_bytes", 0), 2 * hbuf[0].numel() * 8)
        members = reader.open(names)
        pool = ThreadPoolExecutor(max_workers=1)

        def read(k):
            t0 = time.perf_counter()
            arr = hbuf[k % 2].numpy()
            off = read_rows(members, plan[k][1], arr)
            if k == len(plan) - 1:
                for m in members:
                    m.finish()
            arr[off] = 1.0
            stats["read_s"] += time.perf_counter() - t0

        fut = pool.submit(read, 0)
    try:
        for k, (a, n) in enumerate(plan):
            cnt = per_row * n + 1
            err = None
            e0 = torch.cuda.Event(enable_timing=True)
            if rank == 0:
                t0 = time.perf_counter()
                try:
                    fut.result()
                except Exception as e:      # (every rank must still take part in this chunk's broadcast)
                    err = e
                    hbuf[k % 2][cnt - 1] = 0.0
                stats["wait_s"] += time.perf_counter() - t0
                e0.record()
                dbuf[:cnt].copy_(hbuf[k % 2][:cnt], non_blocking=True)
                # hbuf[(k+1) % 2] held chunk k-1, whose copy has finished (plb_unpack_rows synchronised since)
                if err is None and k + 1 < len(plan):
                    fut = pool.submit(read, k + 1)
            else:
                e0.record()
            ctx.call("plb_comm_from_root", dbuf.data_ptr(), cnt)
            if err is not None:
                raise err
            if world > 1 and rank != 0 and float(dbuf[cnt - 1].item()) != 1.0:
                raise ValueError("%s: rank 0 could not read the rows [%d, %d)" % (path, a, a + n))
            views, off = {}, 0
            for name in names:
                views[name] = dbuf[off:off + n * widths[name]].view(n, widths[name])
                off += n * widths[name]
            yield a, n, views
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            stats["events"].append((e0, e1))
    finally:
        if pool is not None:
            pool.shutdown(wait=True)
        for m in members:
            m.close()


def read_snapshot(prefix, it, o, device=None, stats=None):
    """The state written by `write_snapshot` (or by the reference's pylamp2.py:637-650) to `<prefix>griddata.<it>.npz`
    and `<prefix>tracs.<it>.npz`, as a `driver.State` that `driver.timestep(s, o)` continues.  Collective over the
    ranks of the device's context communicator; only rank 0 opens files.

    Restored: nx, L and the grids (the file's axes must be exactly make_grids(nx, L)), it = tstep,
    totaltime = time, newvel / newpres / newtemp (whole planes on every rank), the markers this rank keeps -- all
    rows on one rank; with several ranks the rows of its slab (o.marker_ownership="slab", the migration's owner
    rule) or the file rows [r*M//W, (r+1)*M//W) ("index") -- as tr_x and 13 distinct columns, and trac_vel when tr_v
    has a row per marker (otherwise None: markers were injected after the last advection).  Everything else is as
    in a fresh State: the first step rebuilds the grid fields from the markers (the file's rho is checked for its
    shape only) and starts its solves cold.  Malformed files raise ValueError naming the file and member.
    `stats` (a dict) receives rank 0's timings: read_s (zip reads), wait_s, device_ms, chunks, bytes, pinned_bytes,
    device_buffer_bytes."""
    from .driver import State
    from .migrate import empty_rows, slab_bounds
    ctx = _lib.default_context(device)
    rank, world = ctx.comm_info()
    dev = ctx.torch_device
    st = {"read_s": 0.0, "wait_s": 0.0, "device_ms": 0.0, "chunks": 0, "bytes": 0, "pinned_bytes": 0,
          "device_buffer_bytes": 0, "events": []}
    gpath, tpath = "%sgriddata.%d.npz" % (prefix, it), "%stracs.%d.npz" % (prefix, it)
    # rank 0 checks both files' headers; every rank gets [ok, nz, nxx, Lz, Lx, M, Mv, tstep, time]
    head = torch.zeros(9, dtype=torch.float64, device=dev)
    g, reader, err = None, None, None
    if rank == 0:
        try:
            g = read_griddata(gpath)
            reader = TracsReader(tpath)
            head = torch.tensor([1.0, g["nx"][0], g["nx"][1], g["L"][0], g["L"][1], reader.M, reader.Mv,
                                 float(g["tstep"]), float(g["time"])], dtype=torch.float64, device=dev)
        except Exception as e:      # (the other ranks learn of it through the broadcast)
            err = e
    ctx.call("plb_comm_from_root", head.data_ptr(), head.numel())
    if err is not None:
        raise err
    h = head.tolist()
    if h[0] != 1.0:
        raise ValueError("read_snapshot: rank 0 could not read %s / %s" % (gpath, tpath))
    try:
        nx, L = (int(h[1]), int(h[2])), (h[3], h[4])
        M, Mv = int(h[5]), int(h[6])
        planes = torch.empty((4,) + nx, dtype=torch.float64, device=dev)
        if rank == 0:
            for i, k in enumerate(("velz", "velx", "pres", "temp")):
                planes[i].copy_(torch.from_numpy(g[k]))
        ctx.call("plb_comm_from_root", planes.data_ptr(), planes.numel())
        # which rows this rank keeps: the cell-row range [c0, c1) and the file-row window [lo, hi)
        c0, c1, lo, hi = 0, nx[IZ] - 1, 0, M
        if world > 1 and o.marker_ownership == "slab":
            b = slab_bounds(nx[IZ] - 1, world)
            c0, c1 = b[rank], b[rank + 1]
        elif world > 1:
            b = index_split(M, world)
            lo, hi = b[rank], b[rank + 1]
        plan = read_plan(M)
        ncol = TRACS_MEMBERS[1][1]
        count = C.c_longlong(0)
        if c0 > 0 or c1 < nx[IZ] - 1:
            # count pass over tr_x, so that the arrays are allocated once, at their size
            rows = 0
            for a, n, v in _chunks_to_device(ctx, reader, tpath, ["tr_x"], plan, st):
                ctx.call("plb_unpack_rows", n, v["tr_x"].data_ptr(), None, ncol, None, nx[IZ], L[IZ], c0, c1, 0, n,
                         0, 0, None, None, None, C.byref(count))
                rows += count.value
        else:
            rows = hi - lo
        keep_v = Mv == M
        x = empty_rows(rows, (2,), torch.float64, dev)
        cols = [empty_rows(rows, (), torch.float64, dev) for _ in range(ncol)]
        vel = empty_rows(rows, (2,), torch.float64, dev) if keep_v else None
        names = ["tr_x", "tr_f"] + (["tr_v"] if keep_v else [])
        base = 0
        for a, n, v in _chunks_to_device(ctx, reader, tpath, names, plan, st):
            ctx.call("plb_unpack_rows", n, v["tr_x"].data_ptr(), v["tr_f"].data_ptr(), ncol,
                     v["tr_v"].data_ptr() if keep_v else None, nx[IZ], L[IZ], c0, c1, max(lo - a, 0),
                     min(hi - a, n), base, rows, x.data_ptr(), _lib.ptr_array(cols),
                     vel.data_ptr() if keep_v else None, C.byref(count))
            base += count.value
        if base != rows:
            raise ValueError("%s: %d rows for this rank, the count pass found %d" % (tpath, base, rows))
        torch.cuda.synchronize(dev)
    finally:
        if reader is not None:
            reader.close()
    s = State(nx, L, x, cols, device=dev.index)
    s.it, s.totaltime = int(h[7]), h[8]
    s.newvel, s.newpres, s.newtemp = [planes[0], planes[1]], planes[2], planes[3]
    s.trac_vel = vel
    if stats is not None:
        st["device_ms"] = sum(e0.elapsed_time(e1) for e0, e1 in st["events"])
        st["chunks"] = len(st.pop("events"))
        st["bytes"] = (os.path.getsize(gpath) + os.path.getsize(tpath)) if rank == 0 else 0
        stats.update(st)
    return s
