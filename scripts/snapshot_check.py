"""Multi-GPU snapshot check (torchrun, one process per GPU): a few distributed time steps, then
output.write_snapshot with a small chunk size; rank 0 loads the files and compares them bit for bit with every
rank's arrays gathered independently over a gloo group (rank order), and the grids with driver.full_field.
  torchrun --nproc-per-node 2 scripts/snapshot_check.py [ncell] [nsteps] [index|slab] [local]"""
import os, shutil, sys, tempfile, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pylamp_b200 import _lib, driver, output, setups
from pylamp_b200.pylamp_const import TR__ID

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ncell = int(sys.argv[1]) if len(sys.argv) > 1 else 64
nsteps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
ownership = sys.argv[3] if len(sys.argv) > 3 else "index"
slab_local = len(sys.argv) > 4 and sys.argv[4] == "local"
host_group = dist.new_group(backend="gloo")
ctx = _lib.default_context(local)
ctx.init_comm()
nx, L, tr_x, tr_f, opts = setups.convection(ncell=ncell)
M = tr_x.shape[0]
if ownership == "slab":
    from pylamp_b200 import migrate
    b = migrate.slab_bounds(ncell, world)
    ie = np.clip(np.floor(ncell * tr_x[:, 0] / L[0]).astype(int), 0, ncell - 1)
    sel = np.nonzero(np.searchsorted(b[1:-1], ie, side="right") == rank)[0]
else:
    sel = np.arange((rank * M) // world, ((rank + 1) * M) // world)
s = driver.State(nx, L, tr_x[sel], tr_f[sel], device=local)
o = driver.Options(marker_ownership=ownership, slab_local=slab_local, **opts)
for _ in range(nsteps):
    driver.timestep(s, o)
output.CHUNK_BYTES = 8 * 13 * 1000        # many chunks per rank and array
box = [tempfile.mkdtemp(prefix="snapshot_check_") if rank == 0 else None]
dist.broadcast_object_list(box, src=0, group=host_group)
prefix = os.path.join(box[0], "")
stats = output.write_snapshot(s, prefix)
# independent gathers: every rank's marker arrays (rank order) and the assembled grids
mine = [None] * world
dist.gather_object((s.tr_x.cpu().numpy(), s.tr_f_host(), s.trac_vel.cpu().numpy()), mine if rank == 0 else None,
                   dst=0, group=host_group)
F = {k: driver.full_field(s, f).cpu().numpy() for k, f in (("velz", s.newvel[0]), ("velx", s.newvel[1]),
                                                           ("pres", s.newpres), ("rho", s.f_rho), ("temp", s.newtemp))}
ok = True
if rank == 0:
    t = np.load(prefix + "tracs.%d.npz" % nsteps)
    g = np.load(prefix + "griddata.%d.npz" % nsteps)
    for m, name in enumerate(("tr_x", "tr_f", "tr_v")):
        want = np.concatenate([p[m] for p in mine])
        same = t[name].shape == want.shape and t[name].tobytes() == want.tobytes()
        print(name, t[name].shape, "equal" if same else "DIFFERS", flush=True)
        ok = ok and same
    for k, f in F.items():
        same = g[k].shape == f.shape and g[k].tobytes() == f.tobytes()
        print(k, "equal" if same else "DIFFERS", flush=True)
        ok = ok and same
    ids = t["tr_f"][:, TR__ID].astype(np.int64)
    ok = ok and t["tr_f"].shape[0] == M and np.array_equal(np.sort(ids), np.arange(M))
    print("markers", t["tr_f"].shape[0], "of", M, "ranks", [p[0].shape[0] for p in mine], "stats", stats, flush=True)
    t.close(), g.close()
    shutil.rmtree(box[0])
flag = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
if rank == 0:
    print("SNAPSHOT_CHECK", "OK" if flag.item() else "FAILED", ownership, "local" if slab_local else "")
sys.exit(0 if flag.item() else 1)
