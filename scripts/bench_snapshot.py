"""Time output.write_snapshot on the benchmark's cloud (setups.convection_device, bench.py's solver settings) after a
few steps, on one GPU or under torchrun on several (slab-owned markers with slab-local fields, bench.py's multi-GPU
default).  Measurement only: nothing in the test suite depends on these numbers.

  python scripts/bench_snapshot.py [--ncell 4096] [--calls 2] [--out profiles/snapshot_1gpu.json]
  torchrun --nproc-per-node 4 scripts/bench_snapshot.py --out profiles/snapshot_4gpu.json

Per call of write_snapshot: wall time (host clock, ending in a device synchronise), the device part (sum over the
chunks of pack + NCCL + D2H, CUDA events), the host part (CRC32 + file write of the streamed tracs file, and the
np.savez of the grid file), host time spent waiting for chunks, bytes written.  The files go to a temporary
directory that is deleted; the size falls back to 2048^2 when that directory's file system has no room for one
4096^2 snapshot (about 37 GB), and the JSON says so."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def snapshot_bytes(ncell, per_side):
    """Size of one snapshot: markers x (2 + 13 + 2) doubles + 5 grid planes."""
    M = ncell * ncell * per_side * per_side
    return 8 * 17 * M + 5 * 8 * (ncell + 1) ** 2


def card(local):
    """(name, power limit) of the GPU, read in this run."""
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        name, limit = [x.strip() for x in r.stdout.strip().split(",")[:2]]
        return name, limit
    except Exception:
        return torch.cuda.get_device_name(local), "not measured"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ncell", type=int, default=4096)
    ap.add_argument("--per-side", type=int, default=4)
    ap.add_argument("--steps", type=int, default=2, help="time steps before the snapshots")
    ap.add_argument("--calls", type=int, default=2, help="write_snapshot calls (the first one allocates the buffers)")
    ap.add_argument("--dir", default=tempfile.gettempdir(), help="where the temporary snapshot directory goes")
    ap.add_argument("--out", default=None, help="JSON result (default profiles/snapshot_<n>gpu_<ncell>.json)")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import bench
    from pylamp_b200 import _lib, driver, output, setups
    ctx = _lib.default_context(local)
    if world > 1:
        ctx.init_comm()
    # size: what the file system of the snapshot directory can hold (rank 0 decides, every rank follows)
    box = [None, args.ncell, ""]
    if rank == 0:
        box[0] = tempfile.mkdtemp(prefix="bench_snapshot_", dir=args.dir)
        free = shutil.disk_usage(box[0]).free
        if snapshot_bytes(args.ncell, args.per_side) > 0.9 * free and args.ncell > 2048:
            box[1] = 2048
            box[2] = ("%.1f GB free in the snapshot directory, a %d^2 snapshot needs %.1f GB: measured at 2048^2"
                      % (free / 1e9, args.ncell, snapshot_bytes(args.ncell, args.per_side) / 1e9))
    if world > 1:
        dist.broadcast_object_list(box, src=0)
    tmp, ncell, note = box
    nx, L, tr_x, cols, opts = setups.convection_device(ncell=ncell, per_side=args.per_side, device="cuda:%d" % local,
                                                       rank=rank, world=world)
    s = driver.State(nx, L, tr_x, cols, device=local)
    o = driver.Options(**opts)
    o.marker_ownership = "slab" if world > 1 else "index"
    o.heat_rtol, o.stokes_rtol = bench.DEFAULTS["heat_rtol"], bench.DEFAULTS["stokes_rtol"]
    o.stokes_params = bench.stokes_params()
    for _ in range(args.steps):
        driver.timestep(s, o, want_kelem=False)
    torch.cuda.synchronize()
    calls = []
    for c in range(args.calls):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        st = output.write_snapshot(s, os.path.join(tmp, ""))
        wall = time.perf_counter() - t0
        if rank == 0:
            calls.append({"wall_s": round(wall, 3), "device_ms_sum_over_chunks": round(st["device_ms"], 1),
                          "host_tracs_crc32_write_s": round(st["write_s"], 3),
                          "host_griddata_savez_s": round(st["griddata_s"], 3),
                          "host_wait_for_chunks_s": round(st["wait_s"], 3), "chunks": st["chunks"],
                          "bytes_written": st["bytes"], "GB_per_s_wall": round(st["bytes"] / wall / 1e9, 3)})
            print("call", c, calls[-1], flush=True)
            for f in os.listdir(tmp):
                os.remove(os.path.join(tmp, f))
    if rank == 0:
        shutil.rmtree(tmp)
        name, limit = card(local)
        M = ncell * ncell * args.per_side ** 2
        res = {"what": "output.write_snapshot after %d steps of the benchmark cloud" % args.steps,
               "n_gpus": world, "ncell": ncell, "markers": M, "chunk_bytes": output.CHUNK_BYTES,
               "gpu": name, "power_limit": limit, "snapshot_dir_fs_free_GB": round(shutil.disk_usage(args.dir).free / 1e9, 1),
               "note": note or None, "calls": calls,
               "not_measured": "the split of host time between CRC32 and the file write itself; the disk's own rate"}
        out = args.out or os.path.join(ROOT, "profiles", "snapshot_%dgpu_%d.json" % (world, ncell))
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
