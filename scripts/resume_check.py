"""Multi-GPU resume check (torchrun, one process per GPU): driver.load_npz on 2 ranks.
  torchrun --nproc-per-node 2 scripts/resume_check.py slab|one|index
slab : 3 steps on the ranks (slab-owned markers, slab-local fields), a snapshot, read back on the same ranks: every
       rank's arrays bit for bit what it held; 2 more steps of both runs agree (fields 1e-8 relative L2, markers
       matched by TR__ID 1e-10, limiter, counts, kelem).
one  : rank 0 runs 3 steps on one GPU (before the communicator exists) and writes; both ranks read with slab
       ownership: every marker in its rank's slab, the ids those of the file; 2 more steps agree with the one-GPU
       run's 2 more steps.
index: as "one", read with marker_ownership="index": rank r holds the file rows [r*M//W, (r+1)*M//W)."""
import os, shutil, sys, tempfile, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pylamp_b200 import _lib, driver, migrate, output, setups
from pylamp_b200.pylamp_const import IX, IZ, TR__ID

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
mode = sys.argv[1] if len(sys.argv) > 1 else "slab"
host_group = dist.new_group(backend="gloo")
ctx = _lib.default_context(local)
nx, L, tr_x, tr_f, opts = setups.convection(ncell=64)
M = tr_x.shape[0]
output.CHUNK_BYTES = 8 * 13 * 1000        # many chunks
box = [tempfile.mkdtemp(prefix="resume_check_") if rank == 0 else None]
dist.broadcast_object_list(box, src=0, group=host_group)
prefix = os.path.join(box[0], "")
ok = True


def check(cond, what):
    global ok
    if not cond:
        print("rank", rank, "FAILED:", what, flush=True)
        ok = False


def rel(a, b):
    return float(np.linalg.norm((a - b).ravel()) / max(np.linalg.norm(b.ravel()), 1e-300))


def gathered(s):
    """Rank 0: the fields (full planes) and the markers of every rank sorted by id, the total count, the limiter."""
    F = {k: driver.full_field(s, f).cpu().numpy() for k, f in (("vz", s.newvel[IZ]), ("vx", s.newvel[IX]),
                                                               ("P", s.newpres), ("T", s.newtemp))}
    count = s.count.clone()
    if s.ctx.slab is not None:
        dist.all_reduce(count)
    parts = [None] * world
    dist.gather_object((s.cols[TR__ID].cpu().numpy(), s.tr_x.cpu().numpy(), s.kelem.cpu().numpy()),
                       parts if rank == 0 else None, dst=0, group=host_group)
    if rank != 0:
        return None
    ids = np.concatenate([p[0] for p in parts]).astype(np.int64)
    order = np.argsort(ids, kind="stable")
    return {"F": F, "ids": ids[order], "x": np.concatenate([p[1] for p in parts])[order],
            "kelem": np.concatenate([p[2] for p in parts])[order], "count": int(count.sum()), "limiter": s.limiter}


def agree(g, ref, label):
    if rank != 0:
        return
    e = {k: rel(g["F"][k], ref["F"][k]) for k in g["F"]}
    e["x"] = rel(g["x"], ref["x"])
    print(label, {k: "%.1e" % v for k, v in e.items()}, g["limiter"], ref["limiter"], flush=True)
    check(np.array_equal(g["ids"], ref["ids"]), "%s: ids" % label)
    check(all(e[k] <= 1e-8 for k in ("vz", "vx", "P", "T")), "%s: fields %s" % (label, e))
    check(e["x"] <= 1e-10, "%s: markers %s" % (label, e["x"]))
    check(g["limiter"] == ref["limiter"], "%s: limiter" % label)
    check(g["count"] == ref["count"] == M, "%s: counts %d %d" % (label, g["count"], ref["count"]))
    check(np.mean(g["kelem"] == ref["kelem"]) > 0.9999, "%s: kelem" % label)


if mode == "slab":
    ctx.init_comm()
    b = migrate.slab_bounds(nx[IZ] - 1, world)
    ie = np.clip(np.floor((nx[IZ] - 1) * tr_x[:, 0] / L[0]).astype(int), 0, nx[IZ] - 2)
    sel = np.nonzero(np.searchsorted(b[1:-1], ie, side="right") == rank)[0]
    o = driver.Options(marker_ownership="slab", slab_local=True, **opts)
    s = driver.State(nx, L, tr_x[sel], tr_f[sel], device=local)
    for _ in range(3):
        driver.timestep(s, o)
    driver.save_npz(s, prefix)
    r = driver.load_npz(prefix, 3, o, device=local)
    check(r.it == s.it and r.totaltime == s.totaltime, "it / totaltime")
    same = lambda a, c: a.shape == c.shape and torch.equal(a.contiguous().view(torch.uint8), c.contiguous().view(torch.uint8))
    check(same(r.tr_x, s.tr_x) and same(r.trac_vel, s.trac_vel), "tr_x / trac_vel bits")
    check(all(same(p, q) for p, q in zip(r.cols, s.cols)), "columns bits")
    for k, p, q in (("velz", r.newvel[IZ], s.newvel[IZ]), ("pres", r.newpres, s.newpres), ("temp", r.newtemp, s.newtemp)):
        check(same(p, driver.full_field(s, q)), "%s bits" % k)
    print("rank", rank, "markers", r.ntrac, flush=True)
    for _ in range(2):
        driver.timestep(s, o)
        driver.timestep(r, o)
        if rank == 0:
            print("resumed step", r.it, "stokes_iters", r.stats["stokes_iters"], "uninterrupted",
                  s.stats["stokes_iters"], flush=True)
        agree(gathered(r), gathered(s), "step %d" % r.it)
else:
    ref = None
    if rank == 0:           # the one-GPU run: this context has no communicator yet
        o1 = driver.Options(**opts)
        s1 = driver.State(nx, L, tr_x, tr_f, device=local)
        for _ in range(3):
            driver.timestep(s1, o1)
        driver.save_npz(s1, prefix)
        for _ in range(2):
            driver.timestep(s1, o1)
        ref = {"F": {k: f.cpu().numpy() for k, f in (("vz", s1.newvel[IZ]), ("vx", s1.newvel[IX]),
                                                     ("P", s1.newpres), ("T", s1.newtemp))}}
        order = np.argsort(s1.cols[TR__ID].cpu().numpy(), kind="stable")
        ref.update(ids=s1.cols[TR__ID].cpu().numpy().astype(np.int64)[order], x=s1.tr_x.cpu().numpy()[order],
                   kelem=s1.kelem.cpu().numpy()[order], count=int(s1.count.sum()), limiter=s1.limiter)
        del s1
    dist.barrier(group=host_group)
    ctx.init_comm()
    o = driver.Options(marker_ownership="slab" if mode == "one" else "index", slab_local=True, **opts)
    r = driver.load_npz(prefix, 3, o, device=local)
    with np.load(prefix + "tracs.3.npz") as t:
        fx, ff, fv = t["tr_x"], t["tr_f"], t["tr_v"]
    parts = [None] * world
    dist.all_gather_object(parts, r.cols[TR__ID].cpu().numpy(), group=host_group)
    ids = np.concatenate(parts)
    check(np.array_equal(np.sort(ids), np.sort(ff[:, TR__ID])), "ids are the file's")
    if mode == "one":
        check(migrate.check_ownership(r) == 0, "markers outside the rank's slab")
        print("rank", rank, "markers", r.ntrac, "slab", migrate.slab_bounds(nx[IZ] - 1, world)[rank:rank + 2], flush=True)
        for _ in range(2):
            driver.timestep(r, o)
            if rank == 0:
                print("resumed step", r.it, "stokes_iters", r.stats["stokes_iters"], flush=True)
        agree(gathered(r), ref, "step %d (2 ranks resumed from 1)" % r.it)
    else:
        lo, hi = output.index_split(fx.shape[0], world)[rank:rank + 2]
        host = lambda t: t.cpu().numpy()
        check(host(r.tr_x).tobytes() == fx[lo:hi].tobytes(), "tr_x rows [%d, %d)" % (lo, hi))
        check(r.tr_f_host().tobytes() == ff[lo:hi].tobytes(), "tr_f rows [%d, %d)" % (lo, hi))
        check(host(r.trac_vel).tobytes() == fv[lo:hi].tobytes(), "tr_v rows [%d, %d)" % (lo, hi))
        print("rank", rank, "rows", lo, hi, flush=True)
dist.barrier(group=host_group)
if rank == 0:
    shutil.rmtree(box[0])
flag = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
dist.destroy_process_group()
if rank == 0:
    print("RESUME_CHECK", "OK" if flag.item() else "FAILED", mode)
sys.exit(0 if flag.item() else 1)
