"""Time output.read_snapshot on the benchmark's cloud (setups.convection_device, bench.py's solver settings): a
snapshot written by output.write_snapshot after a few steps, then read back, on one GPU or under torchrun on several
(written and read with slab-owned markers).  Measurement only: nothing in the test suite depends on these numbers.

  python scripts/bench_resume.py [--ncell 4096] [--calls 2] [--out profiles/resume_1gpu_4096.json]
  torchrun --nproc-per-node 2 scripts/bench_resume.py

Per call of read_snapshot (the writer's state freed first): wall time (host clock, ending in a device synchronise),
GB/s of file bytes over it, host seconds in the zip reads (CRC32 / inflate + copy into the pinned buffers, in the
reader thread), host seconds waiting for them, the device milliseconds summed over the chunks (H2D + broadcast +
plb_unpack_rows, CUDA events), the pinned host bytes and this rank's device chunk buffer, and the peak of torch's
allocator during the call above what was allocated before it.  Then one time step of the resumed state.  The files
go to a temporary directory that is deleted; the size falls back to 2048^2 when its file system has no room for a
4096^2 snapshot (about 37 GB), and the JSON says so."""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncell", type=int, default=4096)
    ap.add_argument("--per-side", type=int, default=4)
    ap.add_argument("--steps", type=int, default=1, help="time steps before the snapshot")
    ap.add_argument("--calls", type=int, default=2, help="read_snapshot calls (the first one allocates the buffers)")
    ap.add_argument("--dir", default=tempfile.gettempdir(), help="where the temporary snapshot directory goes")
    ap.add_argument("--out", default=None, help="JSON result (default profiles/resume_<n>gpu_<ncell>.json)")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import bench
    from bench_snapshot import card, snapshot_bytes
    from pylamp_b200 import _lib, driver, output, setups
    ctx = _lib.default_context(local)
    if world > 1:
        ctx.init_comm()
    box = [None, args.ncell, ""]
    if rank == 0:
        box[0] = tempfile.mkdtemp(prefix="bench_resume_", dir=args.dir)
        free = shutil.disk_usage(box[0]).free
        if snapshot_bytes(args.ncell, args.per_side) > 0.9 * free and args.ncell > 2048:
            box[1] = 2048
            box[2] = ("%.1f GB free in the snapshot directory, a %d^2 snapshot needs %.1f GB: measured at 2048^2"
                      % (free / 1e9, args.ncell, snapshot_bytes(args.ncell, args.per_side) / 1e9))
    if world > 1:
        dist.broadcast_object_list(box, src=0)
    tmp, ncell, note = box
    prefix = os.path.join(tmp, "")
    nx, L, tr_x, cols, opts = setups.convection_device(ncell=ncell, per_side=args.per_side, device="cuda:%d" % local,
                                                       rank=rank, world=world)
    o = driver.Options(**opts)
    o.marker_ownership = "slab" if world > 1 else "index"
    o.heat_rtol, o.stokes_rtol = bench.DEFAULTS["heat_rtol"], bench.DEFAULTS["stokes_rtol"]
    o.stokes_params = bench.stokes_params()
    s = driver.State(nx, L, tr_x, cols, device=local)
    del tr_x, cols
    for _ in range(args.steps):
        driver.timestep(s, o, want_kelem=False)
    t0 = time.perf_counter()
    wst = output.write_snapshot(s, prefix)
    write_s = time.perf_counter() - t0
    it = s.it
    del s
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    calls, r = [], None
    for c in range(args.calls):
        r = None
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated(local)
        torch.cuda.reset_peak_memory_stats(local)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        st = {}
        r = output.read_snapshot(prefix, it, o, device=local, stats=st)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        peak = torch.cuda.max_memory_allocated(local) - base
        if rank == 0:
            calls.append({"wall_s": round(wall, 3), "GB_per_s_wall": round(st["bytes"] / wall / 1e9, 3),
                          "host_zip_read_s": round(st["read_s"], 3), "host_wait_for_reads_s": round(st["wait_s"], 3),
                          "device_ms_sum_over_chunks": round(st["device_ms"], 1), "chunks": st["chunks"],
                          "bytes_read": st["bytes"], "pinned_host_bytes": st["pinned_bytes"],
                          "device_chunk_buffer_bytes": st["device_buffer_bytes"],
                          "peak_device_bytes_above_start": int(peak), "rank0_markers": r.ntrac})
            print("call", c, calls[-1], flush=True)
    t0 = time.perf_counter()
    driver.timestep(r, o, want_kelem=False)
    torch.cuda.synchronize()
    step_s = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
    if rank == 0:
        shutil.rmtree(tmp)
        name, limit = card(local)
        res = {"what": "output.read_snapshot of a snapshot written after %d steps of the benchmark cloud" % args.steps,
               "n_gpus": world, "ncell": ncell, "markers": ncell * ncell * args.per_side ** 2,
               "chunk_bytes": output.CHUNK_BYTES, "gpu": name,
               "power_limit": limit, "note": note or None, "write_snapshot_wall_s": round(write_s, 3),
               "write_snapshot_bytes": wst["bytes"], "calls": calls,
               "first_step_after_resume": {"wall_s": round(step_s, 3), "stokes_iters": r.stats.get("stokes_iters"),
                                           "heat_iters": r.stats.get("heat_iters")},
               "not_measured": "the split of the zip read time between the disk, CRC32 and the copy into pinned memory"}
        out = args.out or os.path.join(ROOT, "profiles", "resume_%dgpu_%d.json" % (world, ncell))
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
