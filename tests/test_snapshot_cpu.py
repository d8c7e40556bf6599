"""The streaming `.npz` writer of the snapshots (pylamp_b200/output.py) on NumPy chunks, no GPU: the chunk plan
every rank walks, and files that np.load reads back bit for bit as it reads np.savez output."""
import struct
import zipfile

import numpy as np
import pytest

from pylamp_b200 import output

WIDTHS = [w for _, w in output.TRACS_MEMBERS]


def _write(path, per_rank):
    """per_rank[r] = (tr_x, tr_f, tr_v) of rank r: fed through plan_chunks / write_npz_stream as the GPU path is."""
    counts = [[p[m].shape[0] for p in per_rank] for m in range(len(WIDTHS))]
    jobs = output.plan_chunks(counts, WIDTHS)
    chunks = ((m, per_rank[r][m][a:a + n]) for m, r, a, n in jobs)
    members = [(name, (sum(counts[m]), w)) for m, (name, w) in enumerate(output.TRACS_MEMBERS)]
    output.write_npz_stream(path, members, chunks)
    return jobs


def _local_extra_ids(path):
    """Header ids of the extra fields of every member's local file header."""
    out = {}
    with zipfile.ZipFile(path) as zf, open(path, "rb") as f:
        for info in zf.infolist():
            f.seek(info.header_offset)
            head = f.read(30)
            assert head[:4] == b"PK\x03\x04"
            nname, nextra = struct.unpack("<HH", head[26:30])
            f.seek(info.header_offset + 30 + nname)
            extra, ids = f.read(nextra), []
            while len(extra) >= 4:
                hid, size = struct.unpack("<HH", extra[:4])
                ids.append(hid)
                extra = extra[4 + size:]
            out[info.filename] = ids
    return out


def _cloud(rng, M, Mv=None):
    """tr_x, tr_f, tr_v of M markers (tr_v: Mv rows -- markers injected after the advection have none)"""
    f = rng.standard_normal((M, 13))
    f[:, 11] = np.arange(M)
    return rng.random((M, 2)), f, rng.standard_normal((M if Mv is None else Mv, 2))


@pytest.mark.parametrize("rows_per_rank,chunk_rows", [
    ([0], 4),                 # no markers at all
    ([0, 0, 0], 4),
    ([23], 5),                # not a multiple of the chunk
    ([7, 0, 12, 5], 3),       # several ranks, one of them empty
    ([1000, 333], 7),         # many chunks
    ([9], 100),               # one chunk smaller than the buffer
    ([(30, 26), (8, 8)], 4),  # tr_v without rows for the markers injected after the advection
])
def test_streamed_tracs_equal_arrays_bit_for_bit(tmp_path, monkeypatch, rows_per_rank, chunk_rows):
    monkeypatch.setattr(output, "CHUNK_BYTES", 8 * 13 * chunk_rows)
    rng = np.random.default_rng(100 * len(rows_per_rank) + chunk_rows)
    per_rank = [_cloud(rng, *(M if isinstance(M, tuple) else (M,))) for M in rows_per_rank]
    rows = [M[0] if isinstance(M, tuple) else M for M in rows_per_rank]
    path = str(tmp_path / "tracs.1.npz")
    jobs = _write(path, per_rank)
    # tr_f chunks hold `chunk_rows` rows; tr_x / tr_v chunks the same bytes
    assert all(n <= chunk_rows for m, _, _, n in jobs if m == 1)
    assert all(n <= chunk_rows * 13 // 2 for m, _, _, n in jobs if m != 1)
    with np.load(path) as z:
        assert sorted(z.files) == ["tr_f", "tr_v", "tr_x"]
        for m, (name, w) in enumerate(output.TRACS_MEMBERS):
            want = np.concatenate([p[m] for p in per_rank])
            got = z[name]
            assert got.dtype == np.float64 and got.shape == want.shape
            assert got.shape[0] == sum(rows) or m == 2
            assert got.tobytes() == want.tobytes()
    with zipfile.ZipFile(path) as zf:
        assert zf.testzip() is None
        assert all(i.compress_type == zipfile.ZIP_STORED for i in zf.infolist())
    ids = _local_extra_ids(path)
    assert set(ids) == {"tr_x.npy", "tr_f.npy", "tr_v.npy"}
    assert all(0x0001 in v for v in ids.values()), ids          # ZIP64 extended information


def test_streamed_members_match_np_savez(tmp_path, monkeypatch):
    """Same members, same .npy headers and payload bytes as np.savez of the whole arrays."""
    monkeypatch.setattr(output, "CHUNK_BYTES", 8 * 13 * 4)
    rng = np.random.default_rng(5)
    per_rank = [_cloud(rng, 10), _cloud(rng, 3)]
    path, ref = str(tmp_path / "a.npz"), str(tmp_path / "b.npz")
    _write(path, per_rank)
    np.savez(ref, **{name: np.concatenate([p[m] for p in per_rank])
                     for m, (name, _) in enumerate(output.TRACS_MEMBERS)})
    with zipfile.ZipFile(path) as a, zipfile.ZipFile(ref) as b:
        assert a.namelist() == b.namelist()
        for n in a.namelist():
            assert a.read(n) == b.read(n)


def test_plan_walks_members_then_ranks_then_chunks(monkeypatch):
    monkeypatch.setattr(output, "CHUNK_BYTES", 8 * 13 * 2)
    jobs = output.plan_chunks([[3, 0, 2], [3, 0, 2], [2, 1, 2]], [2, 13, 2])
    assert jobs == [(0, 0, 0, 3), (0, 2, 0, 2),
                    (1, 0, 0, 2), (1, 0, 2, 1), (1, 2, 0, 2),
                    (2, 0, 0, 2), (2, 1, 0, 1), (2, 2, 0, 2)]


def test_short_or_overflowing_member_is_an_error(tmp_path):
    members = [("tr_x", (3, 2))]
    with pytest.raises(ValueError):
        output.write_npz_stream(str(tmp_path / "s.npz"), members, [(0, np.zeros((2, 2)))])
    with pytest.raises(ValueError):
        output.write_npz_stream(str(tmp_path / "o.npz"), members, [(0, np.zeros((4, 2)))])
