"""The snapshot reader's host side (pylamp_b200/output.py), no GPU: the streaming member reader against np.load on
files from np.savez, np.savez_compressed and the streaming writer; the rejections of malformed files; the read chunk
plan and the index-mode split."""
import io
import zipfile

import numpy as np
import pytest

from pylamp_b200 import output
from pylamp_b200.setups import make_grids


def _cloud(rng, M, Mv=None):
    f = rng.standard_normal((M, 13))
    f[:, 11] = np.arange(M)
    return rng.random((M, 2)), f, rng.standard_normal((M if Mv is None else Mv, 2))


def _save(path, how, x, f, v):
    if how == "savez":
        np.savez(path, tr_x=x, tr_f=f, tr_v=v)
    elif how == "savez_compressed":
        np.savez_compressed(path, tr_x=x, tr_f=f, tr_v=v)
    else:
        arrays = (x, f, v)
        members = [(name, a.shape) for (name, _), a in zip(output.TRACS_MEMBERS, arrays)]
        output.write_npz_stream(path, members, [(m, a) for m, a in enumerate(arrays)])


def _stream(path):
    """tr_x, tr_f (in lockstep over read_plan) and tr_v as the reader's members deliver them, chunk by chunk."""
    with output.TracsReader(path) as r:
        out = {"tr_x": [], "tr_f": [], "tr_v": []}
        for names, M in ((["tr_x", "tr_f"], r.M), (["tr_v"], r.Mv)):
            members = r.open(names)
            for a, n in output.read_plan(M):
                buf = np.full(n * sum(m.width for m in members) + 3, 7.0)
                off = output.read_rows(members, n, buf)
                assert off == buf.size - 3 and np.all(buf[off:] == 7.0)      # nothing written beyond the rows
                k = 0
                for m in members:
                    out[m.name].append(buf[k:k + n * m.width].reshape(n, m.width))
                    k += n * m.width
            for m in members:
                m.finish()
                m.close()
        return r.M, r.Mv, {k: np.concatenate(v) if v else np.zeros((0, w)) for (k, w), v in
                           zip(output.TRACS_MEMBERS, out.values())}


@pytest.mark.parametrize("how", ["savez", "savez_compressed", "stream"])
@pytest.mark.parametrize("M,Mv,chunk_rows", [(23, 23, 5), (0, 0, 4), (1, 1, 4), (1000, 1000, 7), (30, 26, 4),
                                             (9, 9, 100)])
def test_streamed_members_equal_np_load(tmp_path, monkeypatch, how, M, Mv, chunk_rows):
    monkeypatch.setattr(output, "CHUNK_BYTES", 8 * 13 * chunk_rows)
    monkeypatch.setattr(output, "READ_PIECE", 40)          # zip reads that split rows and doubles
    rng = np.random.default_rng(M + 7 * chunk_rows)
    x, f, v = _cloud(rng, M, Mv)
    path = str(tmp_path / "tracs.3.npz")
    _save(path, how, x, f, v)
    if how == "savez_compressed":
        with zipfile.ZipFile(path) as zf:
            assert all(i.compress_type == zipfile.ZIP_DEFLATED for i in zf.infolist())
    gotM, gotMv, got = _stream(path)
    assert (gotM, gotMv) == (M, Mv)
    with np.load(path) as z:
        for name, _ in output.TRACS_MEMBERS:
            assert got[name].shape == z[name].shape and got[name].tobytes() == z[name].tobytes(), name


def test_read_plan_and_index_split(monkeypatch):
    monkeypatch.setattr(output, "CHUNK_BYTES", 8 * 13 * 4 + 5)
    assert output.read_plan(0) == []
    assert output.read_plan(1) == [(0, 1)]
    assert output.read_plan(10) == [(0, 4), (4, 4), (8, 2)]
    monkeypatch.setattr(output, "CHUNK_BYTES", 8)          # less than a row: one row per chunk
    assert output.read_plan(3) == [(0, 1), (1, 1), (2, 1)]
    assert output.index_split(10, 1) == [0, 10]
    assert output.index_split(10, 2) == [0, 5, 10]
    assert output.index_split(10, 3) == [0, 3, 6, 10]
    assert output.index_split(2, 3) == [0, 0, 1, 2]
    for M in (0, 1, 7, 1001):
        for W in (1, 2, 3):
            b = output.index_split(M, W)
            assert b[0] == 0 and b[-1] == M and all(b[r] == (r * M) // W for r in range(W + 1))


def _npy(arr=None, header=None, payload=None):
    """Bytes of a .npy member: np.save of `arr`, or a format 1.0 header dict + raw payload."""
    b = io.BytesIO()
    if arr is not None:
        np.save(b, arr)
    else:
        np.lib.format.write_array_header_1_0(b, header)
        b.write(payload)
    return b.getvalue()


def _zip(path, members):
    with zipfile.ZipFile(path, "w") as zf:
        for name, data in members.items():
            zf.writestr(name + ".npy", data)


def _tracs(rng, M=6, Mv=None):
    x, f, v = _cloud(rng, M, Mv)
    return {"tr_x": _npy(x), "tr_f": _npy(f), "tr_v": _npy(v)}


def _read_all(path):
    with output.TracsReader(path) as r:
        members = r.open(["tr_x", "tr_f", "tr_v"])
        buf = np.empty(17 * max(r.M, r.Mv))
        output.read_rows(members[:2], r.M, buf)
        output.read_rows(members[2:], r.Mv, buf)
        for m in members:
            m.finish()


@pytest.mark.parametrize("case,member", [("float32", "tr_x"), ("fortran", "tr_f"), ("width12", "tr_f"),
                                         ("missing", "tr_v"), ("rows", "tr_f"), ("bigendian", "tr_v"),
                                         ("onedim", "tr_x")])
def test_malformed_tracs_headers_are_rejected(tmp_path, case, member):
    rng = np.random.default_rng(1)
    m = _tracs(rng)
    x, f, v = _cloud(rng, 6)
    if case == "float32":
        m["tr_x"] = _npy(x.astype(np.float32))
    elif case == "fortran":
        m["tr_f"] = _npy(np.asfortranarray(f))
    elif case == "width12":
        m["tr_f"] = _npy(f[:, :12].copy())
    elif case == "missing":
        del m["tr_v"]
    elif case == "rows":
        m["tr_f"] = _npy(f[:5].copy())
    elif case == "bigendian":
        m["tr_v"] = _npy(v.astype(">f8"))
    elif case == "onedim":
        m["tr_x"] = _npy(x[:, 0].copy())
    path = str(tmp_path / "tracs.1.npz")
    _zip(path, m)
    with pytest.raises(ValueError) as e:
        output.TracsReader(path)
    assert path in str(e.value) and ("member %s" % member) in str(e.value), str(e.value)


@pytest.mark.parametrize("member", ["tr_x", "tr_f", "tr_v"])
def test_truncated_or_corrupt_member_is_an_error(tmp_path, member):
    rng = np.random.default_rng(2)
    x, f, v = _cloud(rng, 6)
    arrays = {"tr_x": x, "tr_f": f, "tr_v": v}
    # truncated: the header says 6 rows, the payload holds less
    m = {k: _npy(a) for k, a in arrays.items()}
    a = arrays[member]
    head = {"descr": "<f8", "fortran_order": False, "shape": a.shape}
    m[member] = _npy(header=head, payload=a.tobytes()[:-8])
    short = str(tmp_path / "short.npz")
    _zip(short, m)
    with pytest.raises(ValueError) as e:
        _read_all(short)
    assert short in str(e.value) and ("member %s" % member) in str(e.value), str(e.value)
    # longer than the header says
    m[member] = _npy(header=head, payload=a.tobytes() + b"\0" * 8)
    long_ = str(tmp_path / "long.npz")
    _zip(long_, m)
    with pytest.raises(ValueError) as e:
        _read_all(long_)
    assert ("member %s" % member) in str(e.value)
    # corrupt: one payload byte flipped in a stored and in a deflated file (CRC32 check)
    for comp in (zipfile.ZIP_STORED, zipfile.ZIP_DEFLATED):
        good = str(tmp_path / "good.npz")
        with zipfile.ZipFile(good, "w", compression=comp) as zf:
            for k, arr in arrays.items():
                zf.writestr(k + ".npy", _npy(arr))
        with zipfile.ZipFile(good) as zf:
            info = zf.getinfo(member + ".npy")
            raw = open(good, "rb").read()
            start = info.header_offset + 30 + len(info.filename) + len(info.extra)
            # a byte inside the member's data (the stored payload's last byte / the deflate stream's middle)
            pos = start + (info.compress_size - 1 if comp == zipfile.ZIP_STORED else info.compress_size // 2)
        bad = bytearray(raw)
        bad[pos] ^= 0x40
        path = str(tmp_path / "bad.npz")
        open(path, "wb").write(bytes(bad))
        with pytest.raises(ValueError) as e:
            _read_all(path)
        assert path in str(e.value) and ("member %s" % member) in str(e.value), str(e.value)


def _griddata(path, nx=(5, 4), L=(2.0, 3.0), **over):
    grid, _ = make_grids(list(nx), list(L))
    d = dict(gridz=grid[0], gridx=grid[1], velz=np.ones(nx), velx=np.ones(nx), pres=np.ones(nx), rho=np.ones(nx),
             temp=np.ones(nx), tstep=3, time=1.5)
    d.update(over)
    d = {k: v for k, v in d.items() if v is not None}
    np.savez(path, **d)


def test_griddata_is_read_and_checked(tmp_path):
    path = str(tmp_path / "griddata.3.npz")
    _griddata(path)
    g = output.read_griddata(path)
    assert g["nx"] == (5, 4) and g["L"] == (2.0, 3.0) and int(g["tstep"]) == 3 and float(g["time"]) == 1.5
    grid, _ = make_grids([5, 4], [2.0, 3.0])
    off = grid[0].copy()
    off[2] = np.nextafter(off[2], 10.0)                    # one ulp away from linspace(0, L, n)
    cases = {"gridz": dict(gridz=off),
             "gridx": dict(gridx=np.linspace(0.5, 3.0, 4)),
             "velz": dict(velz=np.ones((4, 4))),
             "temp": dict(temp=np.ones((5, 4), dtype=np.float32)),
             "rho": dict(rho=None),
             "tstep": dict(tstep=np.array([3])),
             "time": dict(time=None)}
    for member, over in cases.items():
        bad = str(tmp_path / ("griddata_%s.npz" % member))
        _griddata(bad, **over)
        with pytest.raises(ValueError) as e:
            output.read_griddata(bad)
        assert bad in str(e.value) and ("member %s" % member) in str(e.value), str(e.value)
