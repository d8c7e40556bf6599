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
"""
import os
import time
import zipfile

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
